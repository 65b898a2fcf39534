"""Autograd bindings of the per-op C entry points (include/ralenet_b200.h).

Each Function mirrors one reference forward (cited in the header) and calls the hand-written
sm_100a kernels through the C ABI on the current CUDA stream.  Inputs must be CUDA fp32 tensors;
there is no CPU or PyTorch fallback -- anything else raises.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import STRUCTS, CONSTS

RL_F_PRENORM = CONSTS["RL_F_PRENORM"]
RL_F_RESIDUAL = CONSTS["RL_F_RESIDUAL"]
LE_NONE, LE_PARTIAL, LE_DEPTHWISE = CONSTS["RL_LE_NONE"], CONSTS["RL_LE_PARTIAL"], CONSTS["RL_LE_DEPTHWISE"]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _chk(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.RalenetError(
            f"{name} is on {t.device}: ecg_denoise_b200 runs only on a CUDA B200 device (no CPU fallback)")
    if t.dtype != torch.float32:
        raise _lib.RalenetError(f"{name} has dtype {t.dtype}; the sm_100a kernels take float32")
    _lib.check_device(t.device.index if t.device.index is not None else torch.cuda.current_device())
    return t.contiguous()


def _fill(struct_name: str, **kw):
    s = STRUCTS[struct_name]()
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            v = v.data_ptr()
        setattr(s, k, v)
    return s


_PE_CACHE: Dict[Tuple[str, int, int], torch.Tensor] = {}


def pos_table(L: int, C: int, device) -> torch.Tensor:
    """P[:L] of AbsPositionalEncoding (model/transformer.py:172-177), built in fp32 on the host exactly
    like the reference and cached on the device (the reference re-uploads it in every block)."""
    key = (str(device), L, C)
    t = _PE_CACHE.get(key)
    if t is None:
        X = torch.arange(L, dtype=torch.float32).reshape(-1, 1) / torch.pow(
            10000, torch.arange(0, C, 2, dtype=torch.float32) / C)
        P = torch.zeros(L, C)
        P[:, 0::2] = torch.sin(X)
        P[:, 1::2] = torch.cos(X)
        t = P.to(device)
        _PE_CACHE[key] = t
    return t


def _zeros_like_if(t: Optional[torch.Tensor], need: bool):
    return torch.zeros_like(t) if (t is not None and need) else None


# ------------------------------------------------------------------------------------------------
class AttnBlockFn(torch.autograd.Function):
    """TransformerBlock.forward_part1 + residual / MSAttention.forward (model/transformer.py:383-390, 289-323)."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, wq, bq, wkv, bkv, wp, bp, table, H, W, c0, flags):
        x = _chk(x, "x")
        B, L, C = x.shape
        need = any(ctx.needs_input_grad)
        y = torch.empty_like(x)
        q = k = v = o = lse = None
        if need:
            q, k, v, o = (torch.empty_like(x) for _ in range(4))
            lse = torch.empty(B, H, L, device=x.device, dtype=torch.float32)
        pe = pos_table(L, C, x.device) if flags & RL_F_PRENORM else None
        a = _fill("rl_attn_fwd_args", B=B, L=L, C=C, H=H, W=W, c0=c0, flags=flags, x=x, pe=_p(pe),
                  ln_w=_p(ln_w), ln_b=_p(ln_b), wq=wq, bq=_p(bq), wkv=wkv, bkv=_p(bkv), wp=wp, bp=_p(bp),
                  table=_p(table) if W > 0 else None, y=y, q=_p(q), k=_p(k), v=_p(v), o=_p(o), lse=_p(lse))
        _lib.call("ralenet_attn_fwd", a, _stream())
        if need:
            ctx.save_for_backward(x, ln_w, ln_b, wq, bq, wkv, bkv, wp, bp, table, q, k, v, o, lse)
            ctx.meta = (H, W, c0, flags)
        return y

    @staticmethod
    def backward(ctx, g):
        _lib.deterministic_guard("AttnBlockFn backward (parameter gradients accumulated with atomics)")
        x, ln_w, ln_b, wq, bq, wkv, bkv, wp, bp, table, q, k, v, o, lse = ctx.saved_tensors
        H, W, c0, flags = ctx.meta
        B, L, C = x.shape
        g = _chk(g, "grad")
        nig = ctx.needs_input_grad
        dx = torch.empty_like(x)
        dqkv = torch.empty(B, L, 3 * C, device=x.device, dtype=torch.float32)
        u = torch.empty_like(x)
        ln_need = (nig[1] or nig[2]) and ln_w is not None
        d_ln_w, d_ln_b = _zeros_like_if(ln_w, ln_need), _zeros_like_if(ln_b, ln_need)
        d_wq, d_bq = _zeros_like_if(wq, nig[3]), _zeros_like_if(bq, nig[4])
        d_wkv, d_bkv = _zeros_like_if(wkv, nig[5]), _zeros_like_if(bkv, nig[6])
        d_wp, d_bp = _zeros_like_if(wp, nig[7]), _zeros_like_if(bp, nig[8])
        d_table = _zeros_like_if(table, nig[9] and W > 0)
        pe = pos_table(L, C, x.device) if flags & RL_F_PRENORM else None
        a = _fill("rl_attn_bwd_args", B=B, L=L, C=C, H=H, W=W, c0=c0, flags=flags, g=g, x=x, pe=_p(pe),
                  ln_w=_p(ln_w), ln_b=_p(ln_b), wq=wq, wkv=wkv, wp=wp, table=_p(table) if W > 0 else None,
                  q=q, k=k, v=v, o=o, lse=lse, dx=dx, dqkv=dqkv, u=u,
                  d_ln_w=_p(d_ln_w), d_ln_b=_p(d_ln_b), d_wq=_p(d_wq), d_bq=_p(d_bq), d_wkv=_p(d_wkv),
                  d_bkv=_p(d_bkv), d_wp=_p(d_wp), d_bp=_p(d_bp), d_table=_p(d_table))
        _lib.call("ralenet_attn_bwd", a, _stream())
        return (dx if nig[0] else None, d_ln_w, d_ln_b, d_wq, d_bq, d_wkv, d_bkv, d_wp, d_bp, d_table,
                None, None, None, None)


class FFNBlockFn(torch.autograd.Function):
    """TransformerBlock.forward_part2 + residual / Mlp.forward (model/transformer.py:392-395, 149-161)."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, w1, b1, w2, b2, lew, extra, le_mode, flags):
        x = _chk(x, "x")
        B, L, C = x.shape
        need = any(ctx.needs_input_grad)
        y = torch.empty_like(x)
        h = torch.empty(B, L, 4 * C, device=x.device, dtype=torch.float32) if need else None
        if extra is not None:
            extra = _chk(extra, "extra")
        a = _fill("rl_ffn_fwd_args", B=B, L=L, C=C, le_mode=le_mode, flags=flags, x=x, extra=_p(extra),
                  ln_w=_p(ln_w), ln_b=_p(ln_b), w1=w1, b1=_p(b1), w2=w2, b2=_p(b2), lew=_p(lew), y=y, h=_p(h))
        _lib.call("ralenet_ffn_fwd", a, _stream())
        if need:
            ctx.save_for_backward(x, ln_w, ln_b, w1, b1, w2, b2, lew, h)
            ctx.meta = (le_mode, flags)
        return y

    @staticmethod
    def backward(ctx, g):
        _lib.deterministic_guard("FFNBlockFn backward (parameter gradients accumulated with atomics)")
        x, ln_w, ln_b, w1, b1, w2, b2, lew, h = ctx.saved_tensors
        le_mode, flags = ctx.meta
        B, L, C = x.shape
        g = _chk(g, "grad")
        nig = ctx.needs_input_grad
        dx = torch.empty_like(x)
        dh, g2, u = torch.empty_like(h), torch.empty_like(h), torch.empty_like(x)
        ln_need = (nig[1] or nig[2]) and ln_w is not None
        d_ln_w, d_ln_b = _zeros_like_if(ln_w, ln_need), _zeros_like_if(ln_b, ln_need)
        d_w1, d_b1 = _zeros_like_if(w1, nig[3]), _zeros_like_if(b1, nig[4])
        d_w2, d_b2 = _zeros_like_if(w2, nig[5]), _zeros_like_if(b2, nig[6])
        d_lew = _zeros_like_if(lew, nig[7])
        a = _fill("rl_ffn_bwd_args", B=B, L=L, C=C, le_mode=le_mode, flags=flags, g=g, x=x, ln_w=_p(ln_w),
                  ln_b=_p(ln_b), w1=w1, w2=w2, lew=_p(lew), h=h, dx=dx, dh=dh, g2=g2, u=u,
                  d_ln_w=_p(d_ln_w), d_ln_b=_p(d_ln_b), d_w1=_p(d_w1), d_b1=_p(d_b1), d_w2=_p(d_w2),
                  d_b2=_p(d_b2), d_lew=_p(d_lew))
        _lib.call("ralenet_ffn_bwd", a, _stream())
        return (dx if nig[0] else None, d_ln_w, d_ln_b, d_w1, d_b1, d_w2, d_b2, d_lew,
                g if nig[8] else None, None, None)


class PatchFn(torch.autograd.Function):
    """PatchMerging.forward (mode 0) / PatchSeparate.forward + skip (mode 1) (model/transformer.py:440-460, 418-424)."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, w, skip, mode):
        x = _chk(x, "x")
        B, L, C = x.shape
        need = any(ctx.needs_input_grad)
        shape = (B, L // 2, 2 * C) if mode == 0 else (B, 2 * L, C // 2)
        y = torch.empty(shape, device=x.device, dtype=torch.float32)
        u = torch.empty_like(y) if need else None
        if skip is not None:
            skip = _chk(skip, "skip")
        a = _fill("rl_patch_fwd_args", B=B, L=L, C=C, mode=mode, x=x, skip=_p(skip), ln_w=ln_w, ln_b=ln_b, w=w,
                  y=y, u=_p(u))
        _lib.call("ralenet_patch_fwd", a, _stream())
        if need:
            ctx.save_for_backward(x, ln_w, w, u)
            ctx.mode = mode
        return y

    @staticmethod
    def backward(ctx, g):
        _lib.deterministic_guard("PatchFn backward (parameter gradients accumulated with atomics)")
        x, ln_w, w, u = ctx.saved_tensors
        B, L, C = x.shape
        g = _chk(g, "grad")
        nig = ctx.needs_input_grad
        dx = torch.empty_like(x)
        ln_need = nig[1] or nig[2]
        d_ln_w, d_ln_b = _zeros_like_if(ln_w, ln_need), _zeros_like_if(ln_w, ln_need)
        d_w = _zeros_like_if(w, nig[3])
        a = _fill("rl_patch_bwd_args", B=B, L=L, C=C, mode=ctx.mode, g=g, g2=None, x=x, ln_w=ln_w, w=w, u=u,
                  dx=dx, gsum=None, d_ln_w=_p(d_ln_w), d_ln_b=_p(d_ln_b), d_w=_p(d_w))
        _lib.call("ralenet_patch_bwd", a, _stream())
        return dx if nig[0] else None, d_ln_w, d_ln_b, d_w, g if nig[4] else None, None


class StemFn(torch.autograd.Function):
    """conv1 = Conv1d(2,8,3,p1) -> LeakyReLU(0.2) -> BatchNorm1d(8) -> 'b c l -> b l c'
    (model/transformer.py:570-574, 623, 630).  `reduce_fn(t)` all-reduces the small stat tensors in place
    under data parallelism (SyncBN semantics); None for a single process."""

    @staticmethod
    def forward(ctx, x, conv_w, conv_b, bn_w, bn_b, running_mean, running_var, nbt, training, momentum, eps,
                reduce_fn):
        x = _chk(x, "x")
        B, Cin, L = x.shape
        if Cin != 2:
            raise _lib.RalenetError(f"stem expects 2 input channels (model/transformer.py:571), got {Cin}")
        y = torch.empty(B, L, 8, device=x.device, dtype=torch.float32)
        stats = torch.zeros(64, device=x.device, dtype=torch.float32)
        partials = torch.empty(B * 16, device=x.device, dtype=torch.float32)
        a = _fill("rl_stem_args", B=B, L=L, training=int(training), x=x, conv_w=conv_w, conv_b=conv_b, bn_w=bn_w,
                  bn_b=bn_b, running_mean=running_mean, running_var=running_var, num_batches_tracked=_p(nbt),
                  stats=stats, partials=partials, y=y, momentum=momentum, eps=eps)
        if training:
            _lib.call("ralenet_stem_stats", a, _stream())
            if reduce_fn is not None:
                reduce_fn(stats[:17])
        _lib.call("ralenet_stem_apply", a, _stream())
        ctx.save_for_backward(x, conv_w, conv_b, bn_w, running_mean, running_var, stats)
        ctx.meta = (training, eps, reduce_fn)
        return y

    @staticmethod
    def backward(ctx, g):
        _lib.deterministic_guard("StemFn backward (parameter gradients accumulated with atomics)")
        x, conv_w, conv_b, bn_w, running_mean, running_var, stats = ctx.saved_tensors
        training, eps, reduce_fn = ctx.meta
        B, _, L = x.shape
        g = _chk(g, "grad")
        nig = ctx.needs_input_grad
        dx = torch.empty_like(x) if nig[0] else None
        partials = torch.empty(B * 16, device=x.device, dtype=torch.float32)
        d_conv_w, d_conv_b = torch.zeros_like(conv_w), torch.zeros_like(conv_b)
        d_bn_w, d_bn_b = torch.zeros_like(bn_w), torch.zeros_like(bn_w)
        a = _fill("rl_stem_bwd_args", B=B, L=L, training=int(training), g=g, g2=None, x=x, conv_w=conv_w,
                  conv_b=conv_b, bn_w=bn_w, running_mean=running_mean, running_var=running_var, stats=stats,
                  sums=stats[32:].data_ptr(), partials=partials, dx=_p(dx), d_conv_w=d_conv_w, d_conv_b=d_conv_b,
                  d_bn_w=d_bn_w, d_bn_b=d_bn_b, eps=eps)
        _lib.call("ralenet_stem_bwd_stats", a, _stream())
        if training and reduce_fn is not None:
            reduce_fn(stats[32:48])
        _lib.call("ralenet_stem_bwd_apply", a, _stream())
        return (dx, d_conv_w, d_conv_b, d_bn_w, d_bn_b) + (None,) * 7


class HeadFn(torch.autograd.Function):
    """transconv(x_1^T + stem_out) (model/transformer.py:664-667); x, skip token-major [B,L,8] -> [B,2,L]."""

    @staticmethod
    def forward(ctx, x, skip, w, b):
        x = _chk(x, "x")
        skip = _chk(skip, "skip") if skip is not None else None
        B, L, _ = x.shape
        out = torch.empty(B, 2, L, device=x.device, dtype=torch.float32)
        a = _fill("rl_head_fwd_args", B=B, L=L, x=x, skip=_p(skip), w=w, b=b, out=out)
        _lib.call("ralenet_head_fwd", a, _stream())
        ctx.save_for_backward(x, skip, w)
        return out

    @staticmethod
    def backward(ctx, dout):
        _lib.deterministic_guard("HeadFn backward (parameter gradients accumulated with atomics)")
        x, skip, w = ctx.saved_tensors
        B, L, _ = x.shape
        dout = _chk(dout, "grad")
        ds = torch.empty_like(x)
        d_w = torch.zeros_like(w)
        d_b = torch.zeros(2, device=x.device, dtype=torch.float32)
        a = _fill("rl_head_bwd_args", B=B, L=L, dout=dout, x=x, skip=_p(skip), w=w, ds=ds, d_w=d_w, d_b=d_b)
        _lib.call("ralenet_head_bwd", a, _stream())
        return ds, (ds if skip is not None else None), d_w, d_b


class Conv1dFn(torch.autograd.Function):
    """newrale's Conv1d(k=13, pad=6) (+ LeakyReLU) (model/ralenet_12leads.py:684-709)."""

    @staticmethod
    def forward(ctx, x, w, b, act, slope):
        x = _chk(x, "x")
        B, Ci, L = x.shape
        Co, _, K = w.shape
        y = torch.empty(B, Co, L, device=x.device, dtype=torch.float32)
        a = _fill("rl_conv_fwd_args", B=B, L=L, Cin=Ci, Cout=Co, K=K, act=int(act), slope=slope, x=x, w=w, b=_p(b),
                  y=y)
        _lib.call("ralenet_conv1d_fwd", a, _stream())
        ctx.save_for_backward(x, w, b)
        ctx.meta = (act, slope)
        # torch.use_deterministic_algorithms(True) at forward time selects the deterministic backward (as in RalenetFn)
        ctx.det = torch.are_deterministic_algorithms_enabled()
        return y

    @staticmethod
    def backward(ctx, dy):
        if not ctx.det:
            _lib.deterministic_guard("Conv1dFn backward of a forward run without torch.use_deterministic_algorithms(True)")
        x, w, b = ctx.saved_tensors
        act, slope = ctx.meta
        B, Ci, L = x.shape
        Co, _, K = w.shape
        dy = _chk(dy, "grad")
        nig = ctx.needs_input_grad
        dx = torch.empty_like(x) if nig[0] else None
        d_w = torch.zeros_like(w) if nig[1] else None
        d_b = torch.zeros_like(b) if (b is not None and nig[2]) else None
        a = _fill("rl_conv_bwd_args", B=B, L=L, Cin=Ci, Cout=Co, K=K, act=int(act), slope=slope, dy=dy, x=x, w=w,
                  b=_p(b), dx=_p(dx), d_w=_p(d_w), d_b=_p(d_b))
        if ctx.det:
            conv1d_bwd_det(a, conv1d_slab(B, Ci, Co, K, x.device))
        else:
            _lib.call("ralenet_conv1d_bwd", a, _stream())
        return dx, d_w, d_b, None, None


def conv1d_slab(B: int, Ci: int, Co: int, K: int, device) -> torch.Tensor:
    """partial-slab scratch of the deterministic convolution backward (ralenet_conv1d_slab_bytes, float32)."""
    n = int(_lib.load().ralenet_conv1d_slab_bytes(B, Ci, Co, K))
    return torch.empty(n // 4, device=device, dtype=torch.float32)


def conv1d_bwd_det(a, slab: torch.Tensor) -> None:
    """ralenet_conv1d_bwd_det: the convolution backward with window-ordered weight / bias gradient sums."""
    _lib.check(_lib.load().ralenet_conv1d_bwd_det(ctypes.byref(a), slab.data_ptr(), slab.numel() * 4, _stream()))


# ------------------------------------------------------------------------------------------------
class EcaFn(torch.autograd.Function):
    """eca_layer_1d.forward (model/transformer.py:109-113) on (B, L, C) tokens, optionally fused with the block
    residual: y = x * sigmoid(conv_k(mean_t x)) (+ res)."""

    @staticmethod
    def forward(ctx, x, w, res):
        x = _chk(x, "x")
        B, L, C = x.shape
        K = w.numel()
        res = _chk(res, "res") if res is not None else None
        y = torch.empty_like(x)
        s = torch.empty(B, C, device=x.device, dtype=torch.float32)
        a = _fill("rl_eca_fwd_args", B=B, L=L, C=C, K=K, x=x, res=_p(res), w=w, y=y, s=s)
        _lib.call("ralenet_eca_fwd", a, _stream())
        ctx.save_for_backward(x, w, s)
        ctx.has_res = res is not None
        return y

    @staticmethod
    def backward(ctx, g):
        _lib.deterministic_guard("EcaFn backward (parameter gradients accumulated with atomics)")
        x, w, s = ctx.saved_tensors
        B, L, C = x.shape
        g = _chk(g, "grad")
        nig = ctx.needs_input_grad
        dx = torch.empty_like(x)
        d_w = torch.zeros_like(w) if nig[1] else None
        a = _fill("rl_eca_bwd_args", B=B, L=L, C=C, K=w.numel(), g=g, x=x, w=w, s=s, dx=dx, d_w=_p(d_w))
        _lib.call("ralenet_eca_bwd", a, _stream())
        return dx if nig[0] else None, d_w, (g if (ctx.has_res and nig[2]) else None)


def snr_mix(data: torch.Tensor, noise: torch.Tensor, snr_db) -> torch.Tensor:
    """single_snr_noise_add (local_utils/local_utils.py:176-192) for a batch of windows on the GPU:
    out[b] = data[b] + noise[b] * sqrt(mean(data[b]**2) / 10**(snr_db[b]/10) / mean(noise[b]**2)), the means over
    all leads and samples of window b.  `snr_db`: float or (B,) tensor."""
    data, noise = _chk(data, "data"), _chk(noise, "noise")
    if data.shape != noise.shape:
        raise _lib.RalenetError(f"snr_mix: data {tuple(data.shape)} and noise {tuple(noise.shape)} differ")
    B = data.shape[0]
    if not isinstance(snr_db, torch.Tensor):
        snr_db = torch.full((B,), float(snr_db), device=data.device, dtype=torch.float32)
    snr_db = _chk(snr_db, "snr_db")
    if snr_db.numel() != B:
        raise _lib.RalenetError(f"snr_mix: snr_db has {snr_db.numel()} entries for {B} windows")
    out = torch.empty_like(data)
    _lib.check(_lib.load().ralenet_snr_mix(ctypes.c_void_p(data.data_ptr()), ctypes.c_void_p(noise.data_ptr()),
                                           ctypes.c_void_p(snr_db.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                           B, data.numel() // B, ctypes.c_void_p(_stream())))
    return out


# ------------------------------------------------------------------------------------------------
# stand-alone forwards of the helper modules (small_ops.cu) -- fused away inside ralenet.forward, kept callable
class LinearFn(torch.autograd.Function):
    """y = x W^T + b over the last dimension (the nn.Linear inside LinearProjection.forward,
    model/transformer.py:243-244, called on its own)."""

    @staticmethod
    def forward(ctx, x, w, b):
        x = _chk(x, "x")
        K, N = x.shape[-1], w.shape[0]
        M = x.numel() // K
        y = torch.empty(*x.shape[:-1], N, device=x.device, dtype=torch.float32)
        _lib.check(_lib.load().ralenet_linear_fwd(x.data_ptr(), w.data_ptr(), _p(b), y.data_ptr(), M, K, N, _stream()))
        ctx.save_for_backward(x, w)
        ctx.has_bias = b is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        _lib.deterministic_guard("LinearFn backward (parameter gradients accumulated with atomics)")
        x, w = ctx.saved_tensors
        dy = _chk(dy, "grad")
        K, N = x.shape[-1], w.shape[0]
        M = x.numel() // K
        lib = _lib.load()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _lib.check(lib.ralenet_linear_bwd_data(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), M, K, N, _stream()))
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dw = torch.zeros_like(w)
            db = torch.zeros(N, device=x.device, dtype=torch.float32) if ctx.has_bias else None
            _lib.check(lib.ralenet_wgrad(dy.data_ptr(), N, x.data_ptr(), K, M, N, K, dw.data_ptr(), _p(db), _stream()))
        return dx, dw, db


class PeAddFn(torch.autograd.Function):
    """AbsPositionalEncoding.forward (model/transformer.py:179-181): X + P[:, :L] (dropout p = 0)."""

    @staticmethod
    def forward(ctx, x):
        x = _chk(x, "x")
        B, L, C = x.shape
        y = torch.empty_like(x)
        _lib.check(_lib.load().ralenet_pe_add(x.data_ptr(), pos_table(L, C, x.device).data_ptr(), y.data_ptr(), B,
                                              L * C, _stream()))
        return y

    @staticmethod
    def backward(ctx, dy):
        return dy


class PartialConvFn(torch.autograd.Function):
    """PartialConv_1d.forward_split_cat (model/transformer.py:54-59) with dim_conv3 == 1 on a channels-first
    (B, C, L) tensor: channel 0 <- Conv1d(1, 1, 3, padding 1, bias=False), channels 1.. pass through."""

    @staticmethod
    def forward(ctx, x, w):
        x = _chk(x, "x")
        B, C, L = x.shape
        y = torch.empty_like(x)
        _lib.check(_lib.load().ralenet_pconv1(x.data_ptr(), w.data_ptr(), y.data_ptr(), B, C, L, 0, _stream()))
        ctx.save_for_backward(x, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        _lib.deterministic_guard("PartialConvFn backward (parameter gradients accumulated with atomics)")
        x, w = ctx.saved_tensors
        dy = _chk(dy, "grad")
        B, C, L = x.shape
        lib = _lib.load()
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _lib.check(lib.ralenet_pconv1(dy.data_ptr(), w.data_ptr(), dx.data_ptr(), B, C, L, 1, _stream()))
        if ctx.needs_input_grad[1]:
            dw = torch.zeros_like(w)
            _lib.check(lib.ralenet_pconv1_wgrad(dy.data_ptr(), x.data_ptr(), dw.data_ptr(), B, C, L, _stream()))
        return dx, dw


def mse_loss_metrics(pred: torch.Tensor, target: torch.Tensor, want_grad: bool = True, gscale: float = 1.0,
                     global_numel: Optional[int] = None, weight: Optional[torch.Tensor] = None,
                     partials: Optional[torch.Tensor] = None):
    """Fused F.mse_loss (denoise_train.py:53) + its gradient + per-window RMSE / SNR
    (local_utils/evaluate.py:27-29, 49-51).  Returns (loss[1], dout or None, rmse[B], snr[B]).
    partials: optional float32 [B] scratch; with it the per-window sums are added to the loss in window order
    (bit-reproducible) instead of with atomics.  Under torch.use_deterministic_algorithms(True) one is allocated."""
    pred, target = _chk(pred, "pred"), _chk(target, "target")
    B = pred.shape[0]
    if partials is None and torch.are_deterministic_algorithms_enabled():
        partials = torch.empty(B, device=pred.device, dtype=torch.float32)
    per = pred.numel() // B
    loss = torch.zeros(1, device=pred.device, dtype=torch.float32)
    dout = torch.empty_like(pred) if want_grad else None
    rmse = torch.empty(B, device=pred.device, dtype=torch.float32)
    snr = torch.empty(B, device=pred.device, dtype=torch.float32)
    n = pred.numel() if global_numel is None else global_numel
    a = _fill("rl_mse_args", B=B, per=per, pred=pred, target=target, weight=_p(weight), dout=_p(dout), loss=loss,
              rmse=rmse, snr=snr, inv_count=1.0 / n, gscale=gscale, partials=_p(partials))
    _lib.call("ralenet_mse", a, _stream())
    return loss, dout, rmse, snr


def adam_flat(p, g, m, v, step, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, gscale=1.0):
    """torch.optim.Adam defaults (denoise_train.py:24) over flat fp32 buffers; `step` is either a python int
    (1-based) or a device int32 tensor incremented by the call (CUDA-graph friendly)."""
    lib = _lib.load()
    if isinstance(step, torch.Tensor):
        _lib.check(lib.ralenet_adam_dev(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr,
                                        betas[0], betas[1], eps, step.data_ptr(), gscale, _stream()))
    else:
        _lib.check(lib.ralenet_adam(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr,
                                    betas[0], betas[1], eps, int(step), gscale, _stream()))
