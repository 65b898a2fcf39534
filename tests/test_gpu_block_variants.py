"""GPU: every flag, R-wave offset and kernel family of the block entry points, and the sub-module API, against the
float64 block reference (tests/block_reference.py: plain forward formulas, gradients from torch.autograd).

The whole network calls the attention and feed-forward halves only with RL_F_PRENORM | RL_F_RESIDUAL, the centred
R-wave block and q/k/v biases.  The C ABI and the modules accept more: flags 0 / PRENORM / RESIDUAL (MSAttention, Mlp,
TransformerBlock.forward_part1 / forward_part2), any bias-block offset c0 (RelativePositionEmbedding.forward(R_pos)),
qkv_bias=False, `extra` without a residual, and the stand-alone helpers (LinearProjection, AbsPositionalEncoding,
PartialConv_1d, eca_layer_1d).  At the wide stages these paths run through other kernels than the network's:

  * the full flag matrix at B = 3 over the ten stage shapes (256- and 512-sample windows);
  * R-wave offsets c0 in {0, centred, L - W} with W in {1, stage W};
  * at C = 64 / 128 the forward families (tcgen05 tiles, one-window and two-window mma.sync kernels) and the weight-
    gradient families (tcgen05, register tiles, mma.sync groups) at the batch sizes where the selection changes, each
    case checked by the kernel labels of the library's profiler to have run the intended kernels.

Tolerance: |d| <= 1e-3 * (|ref| + rms(ref)) (BASELINE.md section 3).  With RALENET_PARITY_DIR set, the worst error of
every comparison goes to <dir>/parity_block_variants.json.
"""
import ctypes
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import ralenet_oracle as O
from tests import block_reference as R
from tests.block_reference import block_params
from tests.common import rel_rms_err, switches

pytestmark = pytest.mark.gpu
RTOL = 1e-3
REPORT = {}
FLAGS = [0, R.PRENORM, R.RESIDUAL, R.PRENORM | R.RESIDUAL]
FLAG_IDS = ["plain", "prenorm", "resid", "prenorm_resid"]
# (L0, stage): C = 8 << stage, L = L0 >> stage; L * C = 2048 (256-sample windows) or 4096 (512: the two-window kernels)
SHAPES = [(L0, s) for L0 in (256, 512) for s in range(5)]
SHAPE_IDS = [f"L{L0}-s{s}" for L0, s in SHAPES]
WGRAD_FAMILIES = {"default": "wgrad_umma_kernel", "reg2": "wgrad_reg_kernel", "mma": "wgrad_group_kernel"}


def _record(name, err):
    """worst error per comparison and per family (the first path component); written to $RALENET_PARITY_DIR."""
    for key in (name, "worst/" + name.split("/")[0]):
        REPORT[key] = max(float(err), REPORT.get(key, 0.0))
    out_dir = os.environ.get("RALENET_PARITY_DIR")
    if not out_dir:
        return
    try:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "parity_block_variants.json"), "w") as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)
    except OSError:
        pass


def _cmp(name, got, ref, rtol=RTOL):
    assert got is not None, f"{name}: no gradient"
    got, ref = got.detach().double().cpu().reshape(ref.shape), ref.detach().double().cpu()
    err = rel_rms_err(got.numpy(), ref.numpy())
    _record(name, err)
    assert math.isfinite(err) and err <= rtol, f"{name}: rel err {err:.3e} > {rtol}"


def _zero_key_bias_grad(name, d_bkv):
    """softmax is invariant to a per-query shift of the logits: the key half of d_bkv is exactly 0."""
    C = d_bkv.numel() // 2
    g = d_bkv.detach().double().cpu()
    assert float(g[:C].norm()) <= 1e-5 * float(g[C:].norm()) + 1e-12, name


def _rand(rs, *shape, scale=1.0):
    return torch.from_numpy(rs.standard_normal(shape) * scale)


def _dev(t, grad=True):
    return None if t is None else t.float().cuda().requires_grad_(grad)


def _labels(fn):
    """kernel labels of fn() run under the library's profiler (one stream, every launch recorded)."""
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.ops import _stream
    lib = _lib.load()
    n, stride = 8192, 48
    labels, ms = ctypes.create_string_buffer(n * stride), (ctypes.c_float * n)()
    _lib.check(lib.ralenet_profile_begin(ctypes.c_void_p(_stream())))
    try:
        fn()
    finally:
        got = lib.ralenet_profile_end(labels, stride, ms, n)
    assert got > 0
    return [labels.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode() for i in range(got)]


def _expect(labels, want=(), absent=()):
    """every label of `want` ran and none of `absent` did; a name without '<' matches any template tags."""
    have = set(labels) | {l.split("<")[0] for l in labels}
    assert set(want) <= have, (set(want) - have, sorted(set(labels)))
    assert not set(absent) & have, (set(absent) & have, sorted(set(labels)))


class _switch:
    """_lib.set_attn_umma(mode) for the duration of a with-block."""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        from ecg_denoise_b200 import _lib
        self.prev = _lib.set_attn_umma(self.mode)

    def __exit__(self, *exc):
        from ecg_denoise_b200 import _lib
        _lib.set_attn_umma(self.prev)


@pytest.fixture(scope="module")
def ops():
    from ecg_denoise_b200 import ops as _ops
    return _ops


# ------------------------------------------------------------------------------------------------------------------
# attention half (AttnBlockFn)

def _attn_params(rs, C, flags, qkv_bias):
    p = {k: v for k, v in block_params(rs, C, 0).items() if k in R.ATTN_KEYS}
    if not flags & R.PRENORM:
        del p["norm1.weight"], p["norm1.bias"]
    if not qkv_bias:
        del p["attn.qkv_proj.to_q.bias"], p["attn.qkv_proj.to_kv.bias"]
    return p


def _attn_case(ops, tag, B, L, C, flags, qkv_bias=True, W=0, c0=None, seed=0):
    """AttnBlockFn forward + backward against ref_attn: y, dx, every parameter gradient, d_table.  Returns the kernel
    labels of the call."""
    H = C // 4
    rs = np.random.RandomState(seed)
    p = _attn_params(rs, C, flags, qkv_bias)
    table = 0.5 * _rand(rs, 2 * W - 1, H) if W else None
    c0 = ((L - W) // 2 if c0 is None else c0) if W else 0
    x, g = _rand(rs, B, L, C), _rand(rs, B, L, C)
    y_ref, dx_ref, gr = R.attn_fwd_bwd(x, p, H, flags, g, table, W, c0)
    d = {k: _dev(v) for k, v in p.items()}
    xt, tt, gt = _dev(x), _dev(table), g.float().cuda()
    out = {}

    def run():
        out["y"] = ops.AttnBlockFn.apply(xt, *(d.get(k) for k in R.ATTN_KEYS), tt, H, W, c0, flags)
        out["y"].backward(gt)
        torch.cuda.synchronize()
    labels = _labels(run)
    _cmp(f"{tag}/y", out["y"], y_ref)
    _cmp(f"{tag}/dx", xt.grad, dx_ref)
    for k in p:
        _cmp(f"{tag}/d_{k}", d[k].grad, gr[k])
    if W:
        _cmp(f"{tag}/d_table", tt.grad, gr["table"])
    if qkv_bias:
        _zero_key_bias_grad(tag, d["attn.qkv_proj.to_kv.bias"].grad)
    return labels


def _stage(L0, s):
    return L0 >> s, 8 << s, (O.RW_WINDOW[s] if s < 4 else 0)


@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("qkv_bias", [True, False], ids=["qkvb", "noqkvb"])
@pytest.mark.parametrize("L0,s", SHAPES, ids=SHAPE_IDS)
def test_attn_flag_matrix(ops, L0, s, qkv_bias, flags):
    L, C, W = _stage(L0, s)
    _attn_case(ops, f"attention/flags{flags}/L{L0}s{s}/{'qkvb' if qkv_bias else 'noqkvb'}", 3, L, C, flags, qkv_bias,
               W, None, seed=1000 + 10 * s + flags + (5 if qkv_bias else 0) + L0)


@pytest.mark.parametrize("flags", [0, R.PRENORM], ids=["plain", "prenorm"])
@pytest.mark.parametrize("where", ["zero", "centre", "end"])
@pytest.mark.parametrize("W", ["one", "stage"])
@pytest.mark.parametrize("s", [0, 1, 2, 3])
def test_attn_rwave_offsets(ops, s, W, where, flags):
    """the bias block anywhere in [0, L): top-left corner, centre, bottom-right corner; W = 1 is a single diagonal
    element.  At stage 3 (2W - 1) H <= 128 caps W at 4."""
    L, C, Ws = _stage(256, s)
    W = 1 if W == "one" else Ws
    c0 = {"zero": 0, "centre": (L - W) // 2, "end": L - W}[where]
    _attn_case(ops, f"attention/rwave/s{s}/W{W}/c0_{c0}/flags{flags}", 3, L, C, flags, True, W, c0,
               seed=2000 + 100 * s + W + c0 + flags)


# (attention forward mode, B): 2 = tcgen05 tile kernels, 0 = one-window kernels; 0 at B = 515 = two-window groups +
# the odd last window
FWD_FAMILIES = [(2, 1), (2, 37), (0, 1), (0, 37), (0, 515)]
# stage 3 at the three bias-block offsets; stage 4 has no R-wave table
WIDE_OFFSETS = [(3, "zero"), (3, "centre"), (3, "end"), (4, "none")]


@pytest.mark.parametrize("flags", [0, R.PRENORM], ids=["plain", "prenorm"])
@pytest.mark.parametrize("mode,B", FWD_FAMILIES, ids=[f"mode{m}-B{b}" for m, b in FWD_FAMILIES])
@pytest.mark.parametrize("s,where", WIDE_OFFSETS, ids=[f"s{s}-{w}" for s, w in WIDE_OFFSETS])
def test_attn_forward_families_wide(ops, s, where, mode, B, flags):
    L, C, W = _stage(256, s)
    c0 = {"zero": 0, "centre": (L - W) // 2, "end": L - W, "none": 0}[where]
    with _switch(mode):
        labels = _attn_case(ops, f"attention/fwd_mode{mode}/s{s}/B{B}/flags{flags}/c0_{c0}", B, L, C, flags, True, W,
                            c0, seed=3000 + 10 * s + B + flags + c0)
    if mode == 2:
        _expect(labels, [f"attn_fwd_umma<{C}>", f"attn_bwd_kernel<{C}>"], ["attn_fwd_kernel"])
    elif B < 512:
        _expect(labels, [f"attn_fwd_kernel<{C},1>"], ["attn_fwd_umma", f"attn_fwd_kernel<{C},2>"])
    else:
        _expect(labels, [f"attn_fwd_kernel<{C},2>", f"attn_fwd_kernel<{C},1>"], ["attn_fwd_umma"])


def test_attn_two_window_kernel_at_512_samples(ops):
    """L * C = 4096 (512-sample windows): one window over two passes of the per-window kernels (WIN = 2)."""
    labels = _attn_case(ops, "attention/win2/s3", 5, 64, 64, R.PRENORM, True, 4, 7, seed=3900)
    _expect(labels, ["attn_fwd_kernel<64>", "attn_bwd_kernel<64>"], ["attn_fwd_umma", "attn_fwd_kernel<64,1>"])


@pytest.mark.parametrize("flags", [0, R.PRENORM], ids=["plain", "prenorm"])
@pytest.mark.parametrize("family", list(WGRAD_FAMILIES))
@pytest.mark.parametrize("s", [3, 4])
def test_attn_wgrad_families_wide(ops, s, family, flags):
    """the q / k / v weight gradients read the `u` scratch of the data-gradient kernel: x itself without PRENORM."""
    L, C, W = _stage(256, s)
    with switches(family):
        labels = _attn_case(ops, f"attention/wgrad_{family}/s{s}/flags{flags}", 37, L, C, flags, True, W, None,
                            seed=4000 + 10 * s + flags)
    _expect(labels, [WGRAD_FAMILIES[family]], set(WGRAD_FAMILIES.values()) - {WGRAD_FAMILIES[family]})


# ------------------------------------------------------------------------------------------------------------------
# feed-forward half (FFNBlockFn)

def _ffn_case(ops, tag, B, L, C, le, flags, with_extra, seed):
    rs = np.random.RandomState(seed)
    p = {k: v for k, v in block_params(rs, C, le).items() if k not in R.ATTN_KEYS}
    if not flags & R.PRENORM:
        del p["norm2.weight"], p["norm2.bias"]
    x, g = _rand(rs, B, L, C), _rand(rs, B, L, C)
    extra = _rand(rs, B, L, C) if with_extra else None
    y_ref, dx_ref, gr = R.ffn_fwd_bwd(x, p, le, flags, g, extra)
    d = {k: _dev(v) for k, v in p.items()}
    xt, et, gt = _dev(x), _dev(extra), g.float().cuda()
    args = [d.get(k) for k in R.FFN_KEYS] + [d.get(R.LEW_KEY.get(le, ""))]
    out = {}

    def run():
        out["y"] = ops.FFNBlockFn.apply(xt, *args, et, le, flags)
        out["y"].backward(gt)
        torch.cuda.synchronize()
    labels = _labels(run)
    _cmp(f"{tag}/y", out["y"], y_ref)
    _cmp(f"{tag}/dx", xt.grad, dx_ref)
    for k in p:
        _cmp(f"{tag}/d_{k}", d[k].grad, gr[k])
    if with_extra:
        _cmp(f"{tag}/d_extra", et.grad, gr["extra"])
    return labels


@pytest.mark.parametrize("extra", [False, True], ids=["noextra", "extra"])
@pytest.mark.parametrize("le", [0, 1, 2])
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("L0,s", SHAPES, ids=SHAPE_IDS)
def test_ffn_flag_matrix(ops, L0, s, flags, le, extra):
    L, C, _ = _stage(L0, s)
    labels = _ffn_case(ops, f"feed-forward/flags{flags}/L{L0}s{s}/le{le}/{'extra' if extra else 'noextra'}", 3, L, C,
                       le, flags, extra, seed=5000 + 10 * s + 3 * flags + le + (7 if extra else 0) + L0)
    if le == R.LE_DEPTHWISE and L0 == 512 and C <= 16:
        # the depthwise backward of 512-sample windows at the narrow stages leaves the fc1 / fc2 weight gradients to
        # the GEMM launch (with them in the CTA its shared memory would exceed an SM's)
        _expect(labels, [f"ffn_bwd_kernel<{C}>", "wgrad_kernel"])


def _ffn_kernels(C, le):
    """(fwd, bwd) kernel labels of the feed-forward half at 256-sample windows: tcgen05 tiles unless depthwise."""
    k = ("ffn_fwd_kernel", "ffn_bwd_kernel") if le == 2 else ("ffn_fwd_umma", "ffn_bwd_umma")
    return [f"{k[0]}<{C}>", f"{k[1]}<{C}>"]


@pytest.mark.parametrize("le", [0, 1, 2])
@pytest.mark.parametrize("flags", [0, R.PRENORM], ids=["plain", "prenorm"])
@pytest.mark.parametrize("B", [1, 37, 515])
@pytest.mark.parametrize("s", [3, 4])
def test_ffn_wide_batches(ops, s, B, flags, le):
    """C = 64 / 128 with `extra`: le 0 / 1 run the tcgen05 tile kernels (one partial 128-token tile at B = 1, a
    partial last tile at 37 and 515), le 2 the per-window kernels of ffn.cu."""
    L, C, _ = _stage(256, s)
    labels = _ffn_case(ops, f"feed-forward/wide/s{s}/B{B}/flags{flags}/le{le}", B, L, C, le, flags, True,
                       seed=6000 + 10 * s + B + 3 * flags + le)
    other = {"ffn_fwd_kernel", "ffn_bwd_kernel", "ffn_fwd_umma", "ffn_bwd_umma"} - {n.split("<")[0] for n in
                                                                                   _ffn_kernels(C, le)}
    _expect(labels, _ffn_kernels(C, le), other)


@pytest.mark.parametrize("le", [1, 2])
@pytest.mark.parametrize("flags", [0, R.PRENORM], ids=["plain", "prenorm"])
@pytest.mark.parametrize("family", list(WGRAD_FAMILIES))
@pytest.mark.parametrize("s", [3, 4])
def test_ffn_wgrad_families_wide(ops, s, family, flags, le):
    """fc1's weight gradient reads the `u` scratch of the data-gradient kernel (tcgen05 tiles for le 1, ffn.cu for
    le 2): x itself without PRENORM."""
    L, C, _ = _stage(256, s)
    with switches(family):
        labels = _ffn_case(ops, f"feed-forward/wgrad_{family}/s{s}/flags{flags}/le{le}", 37, L, C, le, flags, True,
                           seed=7000 + 10 * s + flags + le)
    _expect(labels, [WGRAD_FAMILIES[family]] + _ffn_kernels(C, le),
            set(WGRAD_FAMILIES.values()) - {WGRAD_FAMILIES[family]})


# ------------------------------------------------------------------------------------------------------------------
# module API: the nn.Modules of the package against the same float64 formulas

def _load(mod, p):
    sd = mod.state_dict()
    mod.load_state_dict({k: (p[k].reshape(v.shape).float() if k in p else v) for k, v in sd.items()}, strict=True)
    return mod.cuda()


def _module_check(tag, mod, call, x, g, ref_fn, p, extra_leaves=None):
    """call(x) through the module vs ref_fn(x, **p, **extra_leaves) in float64: output, dx, every parameter gradient
    of the module (and of the extra leaves: name -> (cuda parameter, float64 value))."""
    extra_leaves = extra_leaves or {}
    xt = _dev(x)
    y = call(xt)
    y.backward(g.float().cuda())
    y_ref, gr = R.with_grads(ref_fn, g, x=x, **p, **{k: v for k, (_, v) in extra_leaves.items()})
    _cmp(f"{tag}/y", y, y_ref)
    _cmp(f"{tag}/dx", xt.grad, gr["x"])
    named = dict(mod.named_parameters())
    assert named, tag
    for k, q in named.items():
        _cmp(f"{tag}/d_{k}", q.grad, gr[k])
    for k, (q, _) in extra_leaves.items():
        _cmp(f"{tag}/d_{k}", q.grad, gr[k])


def _rw(L, W, H, rs):
    from ecg_denoise_b200.model.transformer import RelativePositionEmbedding
    rw = RelativePositionEmbedding(W, L, H)
    table = 0.5 * _rand(rs, 2 * W - 1, H)
    rw.relative_position_bias_table.data = table.float()
    return rw.cuda(), table


def _module_W(s):
    return O.RW_WINDOW[s] if s < 4 else 2        # at C = 128, (2W - 1) H <= 128 allows W = 2


@pytest.mark.parametrize("mask", ["none", "rw", "rpos_zero", "rpos_end"])
@pytest.mark.parametrize("qkv_bias", [True, False], ids=["qkvb", "noqkvb"])
@pytest.mark.parametrize("s", range(5))
def test_module_msattention(s, qkv_bias, mask):
    from ecg_denoise_b200.model.transformer import MSAttention
    L, C, _ = _stage(256, s)
    H, W = C // 4, _module_W(s)
    rs = np.random.RandomState(8000 + 10 * s + (1 if qkv_bias else 0))
    p = {k[5:]: v for k, v in _attn_params(rs, C, 0, qkv_bias).items()}
    m = _load(MSAttention(C, H, qkv_bias=qkv_bias), p)
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    extra, dense, c0 = {}, None, 0
    if mask != "none":
        rw, table = _rw(L, W, H, rs)
        c0 = {"rw": (L - W) // 2, "rpos_zero": 0, "rpos_end": L - W}[mask]
        dense = rw() if mask == "rw" else rw(c0 + W // 2)
        assert dense._rw_src[1] == c0
        extra = {"table": (rw.relative_position_bias_table, table)}

    def ref_fn(x, table=None, **q):
        return R.ref_attn(x, {"attn." + k: v for k, v in q.items()}, H, 0, table, W if mask != "none" else 0, c0)
    _module_check(f"module/msattention/s{s}/{'qkvb' if qkv_bias else 'noqkvb'}/{mask}", m, lambda t: m(t, mask=dense),
                  x, g, ref_fn, p, extra)
    if qkv_bias:
        _zero_key_bias_grad(f"module/msattention/s{s}/{mask}", m.qkv_proj.to_kv.bias.grad)


def test_module_rpos_outside_the_window_raises():
    """a bias block that would leave [0, L) is rejected by the attention entry point, never computed."""
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.model.transformer import MSAttention
    L, C, W = 128, 16, 16
    rs = np.random.RandomState(8100)
    m = MSAttention(C, 4).cuda()
    rw, _ = _rw(L, W, 4, rs)
    x = _rand(rs, 2, L, C).float().cuda()
    for r_pos in (W // 2 - 1, L - W + W // 2 + 1, -5, L + 3):
        with pytest.raises(_lib.RalenetError):
            m(x, mask=rw(r_pos))
        with pytest.raises(_lib.RalenetError):
            with torch.no_grad():
                m(x, mask=rw(r_pos))


def _mlp_params(rs, C, le, use_partial, use_eca):
    mode = R.LE_NONE if not le else (R.LE_PARTIAL if use_partial else R.LE_DEPTHWISE)
    p = {k: v for k, v in block_params(rs, C, mode).items() if k not in R.ATTN_KEYS}
    if use_eca:
        p["mlp.eca.conv.weight"] = _rand(rs, 1, 1, 3, scale=0.7)
    return p, mode


MLP_OPTIONS = [(False, True), (True, True), (True, False)]      # (local_enhence, use_partial)


@pytest.mark.parametrize("use_eca", [False, True], ids=["noeca", "eca"])
@pytest.mark.parametrize("le,use_partial", MLP_OPTIONS, ids=["nole", "partial", "depthwise"])
@pytest.mark.parametrize("s", range(5))
def test_module_mlp(s, le, use_partial, use_eca):
    from ecg_denoise_b200.model.transformer import Mlp
    L, C, _ = _stage(256, s)
    rs = np.random.RandomState(8200 + 10 * s)
    p, mode = _mlp_params(rs, C, le, use_partial, use_eca)
    p = {k[4:]: v for k, v in p.items() if k.startswith("mlp.")}
    m = _load(Mlp(C, 4 * C, local_enhence=le, use_partial=use_partial, use_eca=use_eca), p)
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)

    def ref_fn(x, **q):
        y = R.ref_ffn(x, {"mlp." + k: v for k, v in q.items()}, mode, 0)
        return R.ref_eca(y, q["eca.conv.weight"]) if use_eca else y
    _module_check(f"module/mlp/s{s}/le{mode}/eca{int(use_eca)}", m, m, x, g, ref_fn, p)


@pytest.mark.parametrize("part", ["part1", "part2", "forward"])
@pytest.mark.parametrize("use_eca", [False, True], ids=["noeca", "eca"])
@pytest.mark.parametrize("s", range(5))
def test_module_transformer_block(s, use_eca, part):
    from ecg_denoise_b200.model.transformer import TransformerBlock
    if part == "part1" and use_eca:
        pytest.skip("forward_part1 does not involve the channel gate")
    L, C, _ = _stage(256, s)
    H, W = C // 4, _module_W(s)
    rs = np.random.RandomState(8300 + 10 * s)
    p, mode = _mlp_params(rs, C, True, True, use_eca)
    p.update({k: v for k, v in block_params(rs, C, 0).items() if k in R.ATTN_KEYS})
    blk = _load(TransformerBlock(C, H, local_enhence=True, use_eca=use_eca), p)
    rw, table = _rw(L, W, H, rs)
    c0 = L - W                                          # the bottom-right edge, reached only through R_pos
    mask = rw(c0 + W // 2)
    x, g = _rand(rs, 2, L, C), _rand(rs, 2, L, C)
    call = {"part1": lambda t: blk.forward_part1(t, mask), "part2": blk.forward_part2,
            "forward": lambda t: blk(t, mask)}[part]
    extra = {} if part == "part2" else {"table": (rw.relative_position_bias_table, table)}

    def ffn(t, q, flags):
        if use_eca:
            return R.ref_eca(R.ref_ffn(t, q, mode, R.PRENORM), q["mlp.eca.conv.weight"],
                             t if flags & R.RESIDUAL else None)
        return R.ref_ffn(t, q, mode, flags)

    def ref_fn(x, table=None, **q):
        if part == "part1":
            return R.ref_attn(x, q, H, R.PRENORM, table, W, c0)
        if part == "part2":
            return ffn(x, q, R.PRENORM)
        return ffn(R.ref_attn(x, q, H, R.PRENORM | R.RESIDUAL, table, W, c0), q, R.PRENORM | R.RESIDUAL)
    # parameters the called part does not use keep grad None in the module; compare only those it uses
    used = {"part1": ("norm1.", "attn."), "part2": ("norm2.", "mlp."), "forward": ("",)}[part]
    for k, q in blk.named_parameters():
        q.requires_grad_(k.startswith(used))
    _module_check(f"module/block_{part}/s{s}/eca{int(use_eca)}", _Used(blk), call, x, g, ref_fn, p, extra)


class _Used:
    """the parameters of a module that require grad (the ones the tested call uses)."""

    def __init__(self, mod):
        self.mod = mod

    def named_parameters(self):
        return [(k, q) for k, q in self.mod.named_parameters() if q.requires_grad]


# ------------------------------------------------------------------------------------------------------------------
# helpers: LinearProjection / LinearFn, AbsPositionalEncoding / PeAddFn, PartialConv_1d / PartialConvFn, EcaFn

@pytest.mark.parametrize("shape", ["B3", "B37", "L50"])
@pytest.mark.parametrize("bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("s", range(5))
def test_helper_linear_projection(s, bias, shape):
    """q, k, v of LinearProjection (linear_fwd), dx (linear_bwd_data) and the weight / bias gradients (the single-
    problem ralenet_wgrad path: pick_tile and the SIMT wgrad_kernel) at token counts that are not multiples of the
    tiles: M = 3 L, 37 L and 150."""
    from ecg_denoise_b200.model.transformer import LinearProjection
    L, C, _ = _stage(256, s)
    H = C // 4
    B, N = {"B3": (3, L), "B37": (37, L), "L50": (3, 50)}[shape]
    rs = np.random.RandomState(9000 + 10 * s + (1 if bias else 0))
    p = {"to_q.weight": _rand(rs, C, C, scale=C ** -0.5), "to_kv.weight": _rand(rs, 2 * C, C, scale=C ** -0.5)}
    if bias:
        p.update({"to_q.bias": 0.1 * _rand(rs, C), "to_kv.bias": 0.1 * _rand(rs, 2 * C)})
    m = _load(LinearProjection(C, H, 4, bias=bias), p)
    x = _rand(rs, B, N, C)
    g = _rand(rs, 3 * B * N * C)

    def call(t):
        return torch.cat([v.reshape(-1) for v in m(t)])

    def ref_fn(x, **q):
        qq = R.linear(x, q["to_q.weight"], q.get("to_q.bias")).reshape(B, N, H, 4).transpose(1, 2)
        kv = R.linear(x, q["to_kv.weight"], q.get("to_kv.bias")).reshape(B, N, 2, H, 4).permute(2, 0, 3, 1, 4)
        return torch.cat([qq.reshape(-1), kv[0].reshape(-1), kv[1].reshape(-1)])
    labels = _labels(lambda: _module_check(f"helpers/linear/s{s}/{shape}/{'bias' if bias else 'nobias'}", m, call, x,
                                           g, ref_fn, p))
    _expect(labels, ["linear_fwd_kernel", "linear_bwd_data_kernel", "wgrad_kernel"])


@pytest.mark.parametrize("L0,s", SHAPES, ids=SHAPE_IDS)
def test_helper_pe_add_and_partial_conv(L0, s):
    """AbsPositionalEncoding.forward at every (L, C) and PartialConv_1d.forward on the (4C, L) hidden tensor of every
    stage."""
    from ecg_denoise_b200.model.transformer import AbsPositionalEncoding, PartialConv_1d
    L, C, _ = _stage(L0, s)
    rs = np.random.RandomState(9100 + 10 * s + L0)
    x, g = _rand(rs, 3, L, C), _rand(rs, 3, L, C)
    xt = _dev(x)
    y = AbsPositionalEncoding(C)(xt)
    y.backward(g.float().cuda())
    _cmp(f"helpers/pe_add/L{L0}s{s}/y", y, x + R.pos_table(L, C))
    _cmp(f"helpers/pe_add/L{L0}s{s}/dx", xt.grad, g)

    pc = PartialConv_1d(4 * C, 4 * C, "split_cat")
    w = _rand(rs, 1, 1, 3, scale=0.5)
    pc.partial_conv3.weight.data = w.float()
    pc = pc.cuda()
    xc, gc = _rand(rs, 3, 4 * C, L), _rand(rs, 3, 4 * C, L)

    def ref_fn(x, **q):
        return torch.cat([torch.nn.functional.conv1d(x[:, :1], q["partial_conv3.weight"], padding=1), x[:, 1:]], 1)
    _module_check(f"helpers/pconv/L{L0}s{s}", pc, pc, xc, gc, ref_fn, {"partial_conv3.weight": w})


@pytest.mark.parametrize("with_res", [False, True], ids=["plain", "res"])
@pytest.mark.parametrize("K", [1, 3, 5, 15])
@pytest.mark.parametrize("C", [8, 16, 32, 64, 128, 256])
def test_helper_eca(ops, C, K, with_res):
    """K > C (C = 8, K = 15): every tap of every channel reaches into the zero padding at one end or both."""
    rs = np.random.RandomState(9200 + C + K)
    B, L = 3, 50
    x, g, w = _rand(rs, B, L, C), _rand(rs, B, L, C), _rand(rs, 1, 1, K, scale=0.7)
    res = _rand(rs, B, L, C) if with_res else None
    y_ref, saved = O.eca_fwd(x, w, res)
    dx_ref, dw_ref = O.eca_bwd(g, saved, w)
    xt, wt, rt = _dev(x), _dev(w), _dev(res)
    y = ops.EcaFn.apply(xt, wt, rt)
    y.backward(g.float().cuda())
    tag = f"helpers/eca/C{C}/K{K}/{'res' if with_res else 'plain'}"
    _cmp(f"{tag}/y", y, y_ref)
    _cmp(f"{tag}/dx", xt.grad, dx_ref)
    _cmp(f"{tag}/dw", wt.grad, dw_ref)
    if with_res:
        _cmp(f"{tag}/dres", rt.grad, g)
