"""float64 reference of the general block formulas behind AttnBlockFn / FFNBlockFn (include/ralenet_b200.h), every flag
and option the C ABI accepts, written as plain torch forward expressions.  Gradients come from torch.autograd, so this
reference shares nothing with the kernels nor with the hand-written backward of oracle/ralenet_oracle.py.

  attention:     u = LN1(x * sqrt(C) + P)  (RL_F_PRENORM)  else  u = x
                 y = proj(softmax(0.5 q k^T + bias block at c0) v)  (+ x with RL_F_RESIDUAL)
  feed-forward:  u = LN2(x)  (RL_F_PRENORM)  else  u = x
                 y = fc2(GELU(leconv(GELU(fc1(u)))))  (+ x with RL_F_RESIDUAL)  (+ extra)
  channel gate:  eca(y) = y * sigmoid(conv_K(mean_t y))  (+ res)

Parameters use the reference's state_dict names ("norm1.weight", "attn.qkv_proj.to_q.bias", "mlp.fc1.weight", ...);
a missing bias key means the layer has no bias.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

Tensor = torch.Tensor

PRENORM, RESIDUAL = 1, 2                 # RL_F_PRENORM, RL_F_RESIDUAL
LE_NONE, LE_PARTIAL, LE_DEPTHWISE = 0, 1, 2
HEAD_DIM = 4
LN_EPS = 1e-5

ATTN_KEYS = ("norm1.weight", "norm1.bias", "attn.qkv_proj.to_q.weight", "attn.qkv_proj.to_q.bias",
             "attn.qkv_proj.to_kv.weight", "attn.qkv_proj.to_kv.bias", "attn.proj.weight", "attn.proj.bias")
FFN_KEYS = ("norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias")
LEW_KEY = {LE_PARTIAL: "mlp.leconv.partial_conv3.weight", LE_DEPTHWISE: "mlp.leconv.weight"}


def pos_table(L: int, C: int) -> Tensor:
    """P[:L] of AbsPositionalEncoding: the sinusoid table is built in float32 (as the module builds it), then widened."""
    X = torch.arange(L, dtype=torch.float32).reshape(-1, 1) / torch.pow(
        10000, torch.arange(0, C, 2, dtype=torch.float32) / C)
    P = torch.zeros(L, C, dtype=torch.float32)
    P[:, 0::2] = torch.sin(X)
    P[:, 1::2] = torch.cos(X)
    return P.double()


def layer_norm(z: Tensor, w: Tensor, b: Tensor) -> Tensor:
    mu = z.mean(-1, keepdim=True)
    var = ((z - mu) ** 2).mean(-1, keepdim=True)
    return (z - mu) / torch.sqrt(var + LN_EPS) * w + b


def linear(x: Tensor, w: Tensor, b: Optional[Tensor]) -> Tensor:
    y = x @ w.t()
    return y if b is None else y + b


def gelu(x: Tensor) -> Tensor:
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def bias_block(table: Tensor, W: int, L: int, c0: int) -> Tensor:
    """(H, L, L): table[i - j + W - 1, h] at (c0 + i, c0 + j) for i, j < W, zero elsewhere."""
    H = table.shape[1]
    i = torch.arange(W).view(-1, 1)
    j = torch.arange(W).view(1, -1)
    blk = table[(i - j + W - 1).reshape(-1)].reshape(W, W, H).permute(2, 0, 1)
    return torch.nn.functional.pad(blk, (c0, L - W - c0, c0, L - W - c0))


def ref_attn(x: Tensor, p: Dict[str, Tensor], H: int, flags: int, table: Optional[Tensor] = None, W: int = 0,
             c0: Optional[int] = None) -> Tensor:
    B, L, C = x.shape
    u = x
    if flags & PRENORM:
        u = layer_norm(x * math.sqrt(C) + pos_table(L, C), p["norm1.weight"], p["norm1.bias"])
    q = linear(u, p["attn.qkv_proj.to_q.weight"], p.get("attn.qkv_proj.to_q.bias"))
    kv = linear(u, p["attn.qkv_proj.to_kv.weight"], p.get("attn.qkv_proj.to_kv.bias"))
    heads = lambda t: t.reshape(B, L, H, HEAD_DIM).transpose(1, 2)
    s = heads(q) @ heads(kv[..., :C]).transpose(-1, -2) * HEAD_DIM ** -0.5
    if table is not None and W > 0:
        s = s + bias_block(table, W, L, (L - W) // 2 if c0 is None else c0)
    o = (torch.softmax(s, -1) @ heads(kv[..., C:])).transpose(1, 2).reshape(B, L, C)
    y = linear(o, p["attn.proj.weight"], p.get("attn.proj.bias"))
    return y + x if flags & RESIDUAL else y


def fir3(x: Tensor, w: Tensor) -> Tensor:
    """zero-padded 3-tap cross-correlation along the tokens: y[t] = w0 x[t-1] + w1 x[t] + w2 x[t+1]; x (B, L, n),
    w (n, 3) (one tap triple per channel)."""
    xp = torch.nn.functional.pad(x, (0, 0, 1, 1))
    return w[:, 0] * xp[:, :-2] + w[:, 1] * xp[:, 1:-1] + w[:, 2] * xp[:, 2:]


def ref_ffn(x: Tensor, p: Dict[str, Tensor], le_mode: int, flags: int, extra: Optional[Tensor] = None) -> Tensor:
    u = layer_norm(x, p["norm2.weight"], p["norm2.bias"]) if flags & PRENORM else x
    g1 = gelu(linear(u, p["mlp.fc1.weight"], p.get("mlp.fc1.bias")))
    if le_mode == LE_PARTIAL:          # PartialConv_1d: Conv1d(1, 1, 3) on hidden channel 0, the rest untouched
        w = p[LEW_KEY[LE_PARTIAL]].reshape(1, 3)
        g1 = gelu(torch.cat([fir3(g1[..., :1], w), g1[..., 1:]], -1))
    elif le_mode == LE_DEPTHWISE:      # depthwise Conv1d(4C, 4C, 3, groups=4C)
        g1 = gelu(fir3(g1, p[LEW_KEY[LE_DEPTHWISE]].reshape(-1, 3)))
    y = linear(g1, p["mlp.fc2.weight"], p.get("mlp.fc2.bias"))
    if flags & RESIDUAL:
        y = y + x
    return y if extra is None else y + extra


def ref_eca(x: Tensor, w: Tensor, res: Optional[Tensor] = None) -> Tensor:
    """eca_layer_1d on (B, L, C) tokens: the K-tap zero-padded convolution runs over the channel axis of the token
    means."""
    K = w.numel()
    P = (K - 1) // 2
    m = torch.nn.functional.pad(x.mean(1), (P, P))
    C = x.shape[-1]
    z = sum(w.reshape(-1)[k] * m[:, k:k + C] for k in range(K))
    y = x * torch.sigmoid(z)[:, None, :]
    return y if res is None else y + res


def with_grads(fn, g: Tensor, **inputs):
    """y = fn(**inputs) on float64 leaf copies of every tensor input, backward with g; returns (y, {name: grad})."""
    leaves = {k: (v.detach().double().clone().requires_grad_(True) if isinstance(v, Tensor) else v)
              for k, v in inputs.items()}
    y = fn(**leaves)
    y.backward(g.double())
    return y.detach(), {k: v.grad for k, v in leaves.items() if isinstance(v, Tensor)}


def attn_fwd_bwd(x, p, H, flags, g, table=None, W=0, c0=None):
    """(y, dx, {param name: grad, "table": grad}) of ref_attn."""
    def fn(x, table, **params):
        return ref_attn(x, params, H, flags, table, W, c0)
    y, gr = with_grads(fn, g, x=x, table=table, **p)
    return y, gr.pop("x"), gr


def ffn_fwd_bwd(x, p, le_mode, flags, g, extra=None):
    """(y, dx, {param name: grad, "extra": grad}) of ref_ffn."""
    def fn(x, extra, **params):
        return ref_ffn(x, params, le_mode, flags, extra)
    y, gr = with_grads(fn, g, x=x, extra=extra, **p)
    return y, gr.pop("x"), gr


def _randn(rs, *shape, scale=1.0):
    return torch.from_numpy(rs.standard_normal(shape) * scale)


def block_params(rs, C, le):
    """seeded parameters of one block under the reference's state_dict names: LayerNorm weights near 1, biases
    ~0.1, weights scaled by fan-in; le selects the local-enhancement weight."""
    p = {"norm1.weight": 1 + 0.1 * _randn(rs, C), "norm1.bias": 0.1 * _randn(rs, C),
         "attn.qkv_proj.to_q.weight": _randn(rs, C, C, scale=C ** -0.5), "attn.qkv_proj.to_q.bias": 0.1 * _randn(rs, C),
         "attn.qkv_proj.to_kv.weight": _randn(rs, 2 * C, C, scale=C ** -0.5),
         "attn.qkv_proj.to_kv.bias": 0.1 * _randn(rs, 2 * C),
         "attn.proj.weight": _randn(rs, C, C, scale=C ** -0.5), "attn.proj.bias": 0.1 * _randn(rs, C),
         "norm2.weight": 1 + 0.1 * _randn(rs, C), "norm2.bias": 0.1 * _randn(rs, C),
         "mlp.fc1.weight": _randn(rs, 4 * C, C, scale=C ** -0.5), "mlp.fc1.bias": 0.1 * _randn(rs, 4 * C),
         "mlp.fc2.weight": _randn(rs, C, 4 * C, scale=(4 * C) ** -0.5), "mlp.fc2.bias": 0.1 * _randn(rs, C)}
    if le == LE_PARTIAL:
        p[LEW_KEY[le]] = _randn(rs, 1, 1, 3, scale=0.5)
    elif le == LE_DEPTHWISE:
        p[LEW_KEY[le]] = _randn(rs, 4 * C, 1, 3, scale=0.5)
    return p
