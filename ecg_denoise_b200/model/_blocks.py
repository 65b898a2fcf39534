"""Host-side mirror of the reference's RA-LENet module tree (shared by the three model files).

Same class names, constructor signatures, sub-module attribute names and registration order as
`model/transformer.py` / `model/raletransformer.py` / `model/ralenet_12leads.py` of the reference, so that
`state_dict()` keys, shapes and the default-init RNG order are identical (SURVEY.md section 8b) -- the
parameter containers are stock nn.Linear / nn.Conv1d / nn.LayerNorm / nn.BatchNorm1d.  Only the
`forward` bodies differ: they call the sm_100a kernels of libralenet_b200.so (ops.py / engine.py).
There is no CPU path: forward on a non-CUDA tensor raises.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib, ops
from ..engine import NetPlan, RalenetFn, check_precision, forward_no_grad


def _unsupported(what: str):
    raise NotImplementedError(
        f"{what} is not implemented by the B200 kernels (the reference never enables it on the RA-LENet path)")


class PartialConv_1d(nn.Module):
    """Parameter container of the 'partial' local-enhancement conv (reference model/transformer.py:16-59).
    With n_div == dim it is a Conv1d(1,1,3) on hidden channel 0; the arithmetic is fused into the
    feed-forward kernel (ffn.cu), so calling it directly is not supported."""

    def __init__(self, dim, n_div, forward) -> None:
        super().__init__()
        if forward not in ("slicing", "split_cat"):
            raise NotImplementedError
        self.dim_conv3 = dim // n_div
        self.dim_untouched = dim - self.dim_conv3
        self.partial_conv3 = nn.Conv1d(self.dim_conv3, self.dim_conv3, 3, 1, 1, bias=False)
        if self.dim_conv3 != 1:
            _unsupported(f"PartialConv_1d with {self.dim_conv3} convolved channels")

    def forward(self, x):
        """stand-alone use on a channels-first (B, dim, L) tensor (reference forward_split_cat :54-59 /
        forward_slicing :47-52 -- same arithmetic); inside Mlp.forward the conv is fused into the feed-forward kernel."""
        return ops.PartialConvFn.apply(x, self.partial_conv3.weight)


def drop_path(x, drop_prob: float = 0., training: bool = False, scale_by_keep: bool = True):
    """reference model/transformer.py:62-79.  Stochastic depth is never enabled on the RA-LENet path (every block is
    built with drop_path = 0 -> nn.Identity, :367), so only the pass-through cases exist here."""
    if drop_prob == 0. or not training:
        return x
    _unsupported("stochastic depth (drop_path > 0 in training mode)")


class DropPath(nn.Module):
    def __init__(self, drop_prob: float = 0., scale_by_keep: bool = True):
        super().__init__()
        if drop_prob:
            _unsupported("stochastic depth (drop_path > 0)")
        self.drop_prob, self.scale_by_keep = drop_prob, scale_by_keep

    def forward(self, x):
        return x


class eca_layer_1d(nn.Module):
    """Efficient channel attention on (B, L, C) tokens (reference model/transformer.py:100-113): the Conv1d(1,1,k)
    runs over the channel axis of the per-window channel means.  `res` fuses the block residual."""

    def __init__(self, channels, k_size=3) -> None:
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool1d(1)
        self.conv = nn.Conv1d(1, 1, kernel_size=k_size, padding=(k_size - 1) // 2, bias=False)
        self.sigmoid = nn.Sigmoid()
        self.channels = channels
        self.k_size = k_size

    def forward(self, x, res=None):
        return ops.EcaFn.apply(x, self.conv.weight, res)


class Mlp(nn.Module):
    """Feed-forward with optional local enhancement (reference model/transformer.py:118-161)."""
    _LE_DEFAULT = False

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.,
                 local_enhence=None, use_partial=True, use_eca=False):
        super().__init__()
        if local_enhence is None:
            local_enhence = self._LE_DEFAULT
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        if act_layer is not nn.GELU:
            _unsupported(f"activation {act_layer}")
        if drop:
            _unsupported("dropout > 0")
        if out_features != in_features or hidden_features != 4 * in_features:
            _unsupported("Mlp with hidden != 4*in or out != in")
        self.local_enhence = local_enhence
        self.use_partial = use_partial
        self.use_eca = bool(use_eca)
        # registration order of the reference (:134-140): eca, fc1, act, fc2, drop, leconv
        self.eca = eca_layer_1d(out_features) if use_eca else nn.Identity()
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)
        if local_enhence:
            if use_partial:
                self.leconv = PartialConv_1d(hidden_features, hidden_features, forward="split_cat")
            else:
                self.leconv = nn.Conv1d(hidden_features, hidden_features, kernel_size=3, stride=1, padding=1,
                                        groups=hidden_features, bias=False)

    def _le(self):
        if not self.local_enhence:
            return ops.LE_NONE, None
        if self.use_partial:
            return ops.LE_PARTIAL, self.leconv.partial_conv3.weight
        return ops.LE_DEPTHWISE, self.leconv.weight

    def forward(self, x):
        mode, lew = self._le()
        y = ops.FFNBlockFn.apply(x, None, None, self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias,
                                 lew, None, mode, 0)
        return self.eca(y) if self.use_eca else y


class AbsPositionalEncoding(nn.Module):
    """Sinusoidal table holder (reference model/transformer.py:166-181).  `P` stays a plain attribute (not a
    buffer) like the reference, so state_dict is unchanged; the kernels read a cached device copy."""

    def __init__(self, num_hiddens, dropout=0., max_len=1000):
        super().__init__()
        if dropout:
            _unsupported("dropout > 0")
        self.num_hiddens, self.max_len = num_hiddens, max_len
        pos = torch.arange(max_len, dtype=torch.float32).reshape(-1, 1)
        freq = torch.pow(10000, torch.arange(0, num_hiddens, 2, dtype=torch.float32) / num_hiddens)
        self.P = torch.zeros((1, max_len, num_hiddens))
        self.P[:, :, 0::2] = torch.sin(pos / freq)
        self.P[:, :, 1::2] = torch.cos(pos / freq)

    def forward(self, X):
        """X + P[:, :L] (reference :179-181).  Inside TransformerBlock.forward this is fused into the attention
        kernel together with the sqrt(C) scale and LayerNorm."""
        return ops.PeAddFn.apply(X)


class LinearProjection(nn.Module):
    """q / kv projection parameters (reference model/transformer.py:183-247); fused into MSAttention."""

    def __init__(self, dim, heads=8, dim_head=64, dropout=0., bias=True) -> None:
        super().__init__()
        inner_dim = dim_head * heads
        self.heads = heads
        self.to_q = nn.Linear(dim, inner_dim, bias=bias)
        self.to_kv = nn.Linear(dim, inner_dim * 2, bias=bias)
        self.dim, self.inner_dim = dim, inner_dim
        if dropout > 0:
            _unsupported("dropout > 0")

    def forward(self, x, attn_kv=None):
        """(q, k, v), each (B, heads, L, head_dim) (reference :226-247).  Inside MSAttention.forward the projections
        are fused into the attention kernel."""
        if attn_kv is not None:
            _unsupported("cross attention (attn_kv)")
        B_, N, C = x.shape
        hd = self.inner_dim // self.heads
        q = ops.LinearFn.apply(x, self.to_q.weight, self.to_q.bias)
        kv = ops.LinearFn.apply(x, self.to_kv.weight, self.to_kv.bias)
        q = q.reshape(B_, N, 1, self.heads, hd).permute(2, 0, 3, 1, 4)[0]
        kv = kv.reshape(B_, N, 2, self.heads, hd).permute(2, 0, 3, 1, 4)
        return q, kv[0], kv[1]


class MSAttention(nn.Module):
    """Multi-head self-attention, head_dim 4 (reference model/transformer.py:250-323)."""

    def __init__(self, dim, num_heads, qkv_bias=True, qk_scale=None, attn_drop=0., proj_drop=0.) -> None:
        super().__init__()
        self.dim, self.num_heads = dim, num_heads
        head_dim = dim // num_heads
        if head_dim != 4 or dim not in (8, 16, 32, 64, 128):
            _unsupported(f"MSAttention with dim={dim}, heads={num_heads} (the kernels are built for head_dim 4, "
                         "dim in {8,...,128} -- every stage of RA-LENet)")
        self.scale = qk_scale or head_dim ** -0.5
        if abs(self.scale - 0.5) > 1e-12:
            _unsupported("qk_scale != head_dim**-0.5")
        if attn_drop or proj_drop:
            _unsupported("dropout > 0")
        self.qkv_proj = LinearProjection(dim, num_heads, head_dim, dropout=0, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self.softmax = nn.Softmax(dim=-1)

    def _run(self, x, mask, norm: Optional[nn.LayerNorm], flags: int):
        table, W, c0 = None, 0, 0
        if mask is not None:
            src = getattr(mask, "_rw_src", None)
            if src is None:
                _unsupported("a dense attention mask that was not produced by RelativePositionEmbedding.forward()")
            rw, c0 = src
            table, W = rw.relative_position_bias_table, rw.Length
        qp = self.qkv_proj
        return ops.AttnBlockFn.apply(
            x, norm.weight if norm is not None else None, norm.bias if norm is not None else None,
            qp.to_q.weight, qp.to_q.bias, qp.to_kv.weight, qp.to_kv.bias, self.proj.weight, self.proj.bias,
            table, self.num_heads, W, c0, flags)

    def forward(self, x, attn_kv=None, mask=None):
        if attn_kv is not None:
            _unsupported("cross attention (attn_kv)")
        return self._run(x, mask, None, 0)


class TransformerBlock(nn.Module):
    """Pre-norm block: x + MSA(LN1(x*sqrt(C)+P)) then + Mlp(LN2(.)) (reference model/transformer.py:325-411)."""
    _LE_DEFAULT = False
    _MLP = Mlp

    def __init__(self, dim, num_heads, mlp_ratio=4., qkv_bias=True, qk_scale=None, drop=0., attn_drop=0.,
                 drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm, local_enhence=None, use_partial=True,
                 use_eca=False, pe='abs', use_checkpoint=False, *args, **kwargs) -> None:
        super().__init__()
        if local_enhence is None:
            local_enhence = self._LE_DEFAULT
        if norm_layer is not nn.LayerNorm:
            _unsupported(f"norm_layer {norm_layer}")
        if pe != 'abs':
            _unsupported(f"pe={pe!r}")
        if mlp_ratio != 4.:
            _unsupported("mlp_ratio != 4")
        self.dim, self.num_heads, self.mlp_ratio, self.pe = dim, num_heads, mlp_ratio, pe
        self.use_checkpoint = use_checkpoint     # accepted; the fused backward recomputes what it needs anyway
        self.attn = MSAttention(dim, num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop,
                                proj_drop=drop)
        self.norm1 = norm_layer(dim)
        self.norm2 = norm_layer(dim)
        self.mlp = self._MLP(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop,
                             local_enhence=local_enhence, use_partial=use_partial, use_eca=use_eca)
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.abs_pos_enc = AbsPositionalEncoding(dim)

    def forward_part1(self, x, mask):
        """attention branch WITHOUT the residual (reference :383-390)."""
        return self.attn._run(x, mask, self.norm1, ops.RL_F_PRENORM)

    def forward_part2(self, x):
        """feed-forward branch WITHOUT the residual (reference :392-395)."""
        m = self.mlp
        mode, lew = m._le()
        y = ops.FFNBlockFn.apply(x, self.norm2.weight, self.norm2.bias, m.fc1.weight, m.fc1.bias, m.fc2.weight,
                                 m.fc2.bias, lew, None, mode, ops.RL_F_PRENORM)
        return m.eca(y) if m.use_eca else y

    def forward(self, x, mask=None):
        x = self.attn._run(x, mask, self.norm1, ops.RL_F_PRENORM | ops.RL_F_RESIDUAL)
        m = self.mlp
        mode, lew = m._le()
        if m.use_eca:      # the channel gate sits between fc2 and the residual (reference :158, :410)
            y = ops.FFNBlockFn.apply(x, self.norm2.weight, self.norm2.bias, m.fc1.weight, m.fc1.bias, m.fc2.weight,
                                     m.fc2.bias, lew, None, mode, ops.RL_F_PRENORM)
            return m.eca(y, res=x)
        return ops.FFNBlockFn.apply(x, self.norm2.weight, self.norm2.bias, m.fc1.weight, m.fc1.bias, m.fc2.weight,
                                    m.fc2.bias, lew, None, mode, ops.RL_F_PRENORM | ops.RL_F_RESIDUAL)


class PatchSeparate(nn.Module):
    """(B,L,C) -> (B,2L,C/2): channel halves concatenated along length, LN, Linear (reference :412-424)."""

    def __init__(self, dim, norm_layer=nn.LayerNorm) -> None:
        super().__init__()
        self.dim = dim
        self.reduction = nn.Linear(dim // 2, dim // 2, bias=False)
        self.norm = norm_layer(dim // 2)

    def forward(self, x, skip=None):
        return ops.PatchFn.apply(x, self.norm.weight, self.norm.bias, self.reduction.weight, skip, 1)


class PatchMerging(nn.Module):
    """(B,L,C) -> (B,L/2,2C): neighbour tokens concatenated, LN, Linear (reference :426-460)."""

    def __init__(self, dim, norm_layer=nn.LayerNorm):
        super().__init__()
        self.dim = dim
        self.reduction = nn.Linear(2 * dim, 2 * dim, bias=False)
        self.norm = norm_layer(2 * dim)

    def forward(self, x):
        if x.shape[1] % 2:
            _unsupported("odd sequence length in PatchMerging")
        return ops.PatchFn.apply(x, self.norm.weight, self.norm.bias, self.reduction.weight, None, 0)


class RelativePositionEmbedding(nn.Module):
    """R-wave attention bias: learned (2W-1) x H Toeplitz table on the central W x W block of the L x L
    logits (reference model/transformer.py:508-545).  forward() returns the dense (1,H,L,L) mask for API
    parity; the attention kernel recognises it (attribute `_rw_src`) and reads the table directly."""

    def __init__(self, Length, whole_length, num_heads) -> None:
        super().__init__()
        self.Length, self.whole_length = Length, whole_length
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * Length - 1), num_heads))
        idx = torch.arange(Length).view(-1, 1) - torch.arange(Length).view(1, -1) + (Length - 1)
        self.register_buffer("relative_position_index", idx)

    def parameters_normalize(self):
        self.relative_position_bias_table.data = torch.randn_like(self.relative_position_bias_table.data) * 0.02

    def forward(self, R_pos=None):
        W, L = self.Length, self.whole_length
        c0 = (L - W) // 2 if R_pos is None else int(R_pos) - W // 2
        blk = self.relative_position_bias_table[self.relative_position_index.view(-1)].view(W, W, -1)
        dense = mask_fill(blk.permute(2, 0, 1).contiguous(), c0, L).unsqueeze(0)
        dense._rw_src = (self, c0)
        return dense


def mask_fill(mask, init_len, length):
    """zero-pad a (H, W, W) block to (H, length, length) at offset init_len (reference :547-558)."""
    num_head, window_size, _ = mask.shape
    assert mask.shape[1] == mask.shape[2]
    pad_total = length - window_size
    return F.pad(mask, (init_len, pad_total - init_len, init_len, pad_total - init_len), value=0)


class BasicLayer(nn.Module):
    """`depth` TransformerBlocks sharing one mask (reference model/transformer.py:462-506)."""
    _LE_DEFAULT = False
    _BLOCK = TransformerBlock
    _CHANNELS_FIRST = False

    def __init__(self, dim, depth, num_heads, mlp_ratio=4., qkv_bias=True, qk_scale=None, drop=0., attn_drop=0.,
                 drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm, local_enhence=None, abs_emd=True,
                 downsample=None, upsample=None, use_checkpoint=False) -> None:
        super().__init__()
        if local_enhence is None:
            local_enhence = self._LE_DEFAULT
        self.depth, self.use_checkpoint = depth, use_checkpoint
        self.blocks = nn.ModuleList([
            self._BLOCK(dim=dim, num_heads=num_heads, mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, qk_scale=qk_scale,
                        drop=drop, attn_drop=attn_drop,
                        drop_path=drop_path[i] if isinstance(drop_path, list) else drop_path, act_layer=act_layer,
                        norm_layer=norm_layer, local_enhence=local_enhence, abs_emd=abs_emd,
                        use_checkpoint=use_checkpoint)
            for i in range(depth)])
        self.downsample = downsample
        if self.downsample is not None:
            self.downsample = downsample(dim=dim, norm_layer=norm_layer)

    def forward(self, x, mask=None):
        if self._CHANNELS_FIRST:                      # raletransformer.BasicLayer takes (B, C, L)
            x = x.transpose(1, 2).contiguous()
        for blk in self.blocks:
            x = blk(x, mask)
        if self.downsample is not None:
            x = self.downsample(x)
        if self._CHANNELS_FIRST:
            x = x.transpose(1, 2).contiguous()
        return x


# ------------------------------------------------------------------------------------------------
class _RalenetBase(nn.Module):
    """Shared forward of the three `ralenet` classes: the whole network is one autograd node
    (engine.RalenetFn -> ralenet_net_fwd / ralenet_net_bwd)."""

    def _init_plan(self):
        object.__setattr__(self, "_plan", NetPlan(self))
        object.__setattr__(self, "_anchor", None)

    # the plan holds ctypes pointer tables and device buffers that belong to THIS instance: copies and pickles
    # (copy.deepcopy for EMA / best-model snapshots, torch.save(model)) drop it and rebuild it lazily
    def __getstate__(self):
        state = dict(self.__dict__)
        state.pop("_plan", None)
        state.pop("_anchor", None)
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        self._init_plan()

    @property
    def inference_precision(self) -> str:
        """Precision of the forwards that build no autograd node (under torch.no_grad(), or when neither the input nor
        any parameter requires grad): "fp32" (default) or "tf32".  "tf32" runs the projection and feed-forward GEMMs of
        the 18 blocks as ONE tf32 tensor-core pass on operands rounded to nearest, instead of the 3-pass split that keeps
        them fp32-grade (RL_NET_TF32, include/ralenet_b200.h); the attention core, LayerNorm, GELU, patch layers, stem
        and head are unchanged.  Outputs stay within 1e-2 * (|ref| + rms(ref)) of the fp64 reference.  A forward that is
        recorded for a backward always runs fp32.  torch.backends.cuda.matmul.allow_tf32 has no effect here.  Not part
        of state_dict(); copy.deepcopy and pickling keep it.  Any other value raises ValueError."""
        return self.__dict__.get("_inference_precision", "fp32")

    @inference_precision.setter
    def inference_precision(self, value: str) -> None:
        self.__dict__["_inference_precision"] = check_precision(value)

    def forward(self, x):
        if not x.is_cuda:
            raise _lib.RalenetError(
                "ecg_denoise_b200 ralenet.forward needs a CUDA tensor on a B200: there is no CPU fallback "
                "(move model and data with .cuda(), as denoise_train.py:20,49 does)")
        rg = any(p.requires_grad for p in self.parameters())
        if not torch.is_grad_enabled() or not (rg or x.requires_grad):
            # eval under torch.no_grad() (test_cls.py:166-214, inference.denoise_records): no autograd node,
            # nothing saved for a backward that cannot happen
            return forward_no_grad(self._plan, x)
        a = self._anchor
        if a is None or a.device != x.device or a.requires_grad != rg:
            a = torch.zeros(1, device=x.device, requires_grad=rg)
            object.__setattr__(self, "_anchor", a)
        return RalenetFn.apply(x, a, self._plan)

    def set_data_parallel(self, process_group=None):
        """all-reduce the BatchNorm batch statistics across ranks (SyncBN-equivalent) in forward/backward."""
        import torch.distributed as dist
        self._plan.reduce_fn = (lambda t: dist.all_reduce(t, group=process_group))


def build_ralenet(self, block_layer, norm_layer, le: bool, with_rw: bool, head_first: bool):
    """registers the sub-modules in the reference's order (transformer.py:566-619 / ralenet_12leads.py:568-625 /
    raletransformer.py:565-637)."""
    channels = [2 ** (i + 3) for i in range(5)]
    heads = [2 ** (i + 1) for i in range(5)]
    length = [2 ** (-i + 8) for i in range(5)]
    self.conv1 = nn.Sequential(nn.Conv1d(2, channels[0], kernel_size=3, padding=1), nn.LeakyReLU(0.2),
                               nn.BatchNorm1d(channels[0]))
    if head_first:
        self.transconv = nn.Sequential(nn.Conv1d(channels[0], 2, kernel_size=3, padding=1))
    if with_rw:
        self.rwattn1 = RelativePositionEmbedding(32, length[0], heads[0])
        self.rwattn2 = RelativePositionEmbedding(16, length[1], heads[1])
        self.rwattn3 = RelativePositionEmbedding(8, length[2], heads[2])
        self.rwattn4 = RelativePositionEmbedding(4, length[3], heads[3])
    mk = lambda s: block_layer(channels[s], heads[s], le)
    self.dtransformer1 = mk(0)
    self.pm1 = PatchMerging(channels[0], norm_layer=norm_layer)
    self.dtransformer2 = mk(1)
    self.pm2 = PatchMerging(channels[1], norm_layer=norm_layer)
    self.dtransformer3 = mk(2)
    self.pm3 = PatchMerging(channels[2], norm_layer=norm_layer)
    self.dtransformer34 = mk(3)
    self.pm4 = PatchMerging(channels[3], norm_layer=norm_layer)
    self.transformer = mk(4)
    self.utransformer4 = mk(4)
    self.ps4 = PatchSeparate(channels[4], norm_layer=norm_layer)
    self.utranformer3 = mk(3)
    self.ps3 = PatchSeparate(channels[3], norm_layer=norm_layer)
    self.utransformer2 = mk(2)
    self.ps2 = PatchSeparate(channels[2], norm_layer=norm_layer)
    self.utransformer1 = mk(1)
    self.ps1 = PatchSeparate(channels[1], norm_layer=norm_layer)
    if not head_first:
        self.transconv = nn.Sequential(nn.Conv1d(channels[0], 2, kernel_size=3, padding=1))
    if norm_layer is not nn.LayerNorm:
        _unsupported(f"norm_layer {norm_layer}")
