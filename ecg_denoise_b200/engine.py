"""Whole-network execution of RA-LENet through `ralenet_net_fwd` / `ralenet_net_bwd`.

`NetPlan` keeps, per `ralenet` module instance, what the C side needs: all parameters flattened into ONE
contiguous fp32 buffer (the nn.Parameters become views into it, so `state_dict()`, `load_state_dict()`,
`optim.Adam(model.parameters())` and `torch.save` keep working on the stock Parameters,
SURVEY.md section 8b), a matching flat gradient buffer that the kernels accumulate into and that the
Parameters' `.grad` alias, the pointer tables, the positional tables and the BatchNorm stat scratch.

`RalenetFn` is the autograd node of `ralenet.forward`: one C call per direction instead of ~1300 ATen
dispatches.  Parameter gradients are written straight into the aliased `.grad` views (accumulating,
like autograd does), so a training step costs no per-parameter Python work.
"""
from __future__ import annotations

import ctypes
import os
from typing import Callable, List, Optional

import torch
import torch.nn as nn

from . import _lib
from ._lib import CONSTS, STRUCTS
from .ops import _chk, _stream, pos_table

# forward order of the 9 two-block layers (attribute names are the reference's, typos included)
LAYER_NAMES = ["dtransformer1", "dtransformer2", "dtransformer3", "dtransformer34", "transformer",
               "utransformer4", "utranformer3", "utransformer2", "utransformer1"]


def _blocks_of(layer: nn.Module) -> List[nn.Module]:
    return list(layer.blocks) if hasattr(layer, "blocks") else list(layer)


class NetPlan:
    def __init__(self, net: nn.Module):
        self.net = net
        self.flat: Optional[torch.Tensor] = None
        self.flat_grad: Optional[torch.Tensor] = None
        self.params: List[nn.Parameter] = []
        self.offsets: List[int] = []
        self.P = STRUCTS["rl_net_ptrs"]()
        self.G = STRUCTS["rl_net_ptrs"]()
        self.bn_stats: Optional[torch.Tensor] = None
        self.pe = None
        self.pe_L0 = None
        self.le_mode = 0
        self.reduce_fn: Optional[Callable[[torch.Tensor], None]] = None   # DP all-reduce of BN stats
        self.last_ws_bytes = 0          # size of the workspace the most recent forward used (tests)

    # -- flattening ------------------------------------------------------------------------------
    def _aliased(self) -> bool:
        """every Parameter slot of the network still holds the Parameter object the plan knows, and its storage is
        still its slice of the flat buffer.  Runs before every forward and backward, so it goes through the cached
        (module, name) slots -- ~300 dict lookups and integer compares, 0.1 ms -- instead of walking the module tree
        (net.parameters() costs 1.5 ms per call for the 311 parameters: a third of the drop-in step at 256 windows)."""
        if self.flat is None or not self.params:
            return False
        base = self.flat.data_ptr()
        for (mod, name), q, o in zip(self._slots, self.params, self.offsets):
            if mod._parameters.get(name) is not q or q.data_ptr() != base + 4 * o:
                return False
        return True

    def ensure(self, device: torch.device):
        """(re)build the flat buffers and pointer tables if the parameters moved."""
        if self._aliased() and self.flat.device == device:
            return
        ps = list(self.net.parameters())
        for p in ps:
            if p.dtype != torch.float32:
                raise _lib.RalenetError(f"parameter dtype {p.dtype}: the sm_100a kernels are float32 "
                                        "(the reference is fp32 everywhere, SURVEY.md section 2.1)")
            if p.device != device:
                raise _lib.RalenetError(f"parameter on {p.device} but input on {device}: call model.cuda() first")
        offs, n = [], 0
        for p in ps:
            offs.append(n)
            n += (p.numel() + 3) // 4 * 4              # keep every tensor 16-byte aligned
        flat = torch.zeros(n, device=device, dtype=torch.float32)
        flat_grad = torch.zeros(n, device=device, dtype=torch.float32)
        with torch.no_grad():
            for p, o in zip(ps, offs):
                flat[o:o + p.numel()].copy_(p.detach().reshape(-1))
                old_grad = p.grad
                p.data = flat[o:o + p.numel()].view(p.shape)
                if old_grad is not None:
                    flat_grad[o:o + p.numel()].copy_(old_grad.reshape(-1))
                    p.grad = flat_grad[o:o + p.numel()].view(p.shape)
        self.flat, self.flat_grad, self.params, self.offsets = flat, flat_grad, ps, offs
        self.n_flat = n
        # where each Parameter lives (same order as net.parameters(): named_parameters walks named_modules and
        # de-duplicates shared Parameters the same way)
        slot_of = {}
        for mod in self.net.modules():
            for name, q in mod._parameters.items():
                if q is not None and id(q) not in slot_of:
                    slot_of[id(q)] = (mod, name)
        self._slots = [slot_of[id(q)] for q in ps]
        self._grad_views = None
        self.bn_stats = torch.zeros(64, device=device, dtype=torch.float32)
        self._build_tables()

    def rebind_grad(self, buf: torch.Tensor):
        """move the flat gradient buffer into caller-provided memory (the symmetric buffer of comm.SymmComm, so the
        backward kernels accumulate straight into peer-visible memory); existing gradients are carried over."""
        assert buf.numel() == self.n_flat and buf.dtype == torch.float32 and buf.device == self.flat.device
        if self.flat_grad is not None and buf.data_ptr() == self.flat_grad.data_ptr():
            return
        with torch.no_grad():
            buf.copy_(self.flat_grad)
            old_base = self.flat_grad.data_ptr()
            for p, o in zip(self.params, self.offsets):
                if p.grad is not None and p.grad.data_ptr() == old_base + 4 * o:
                    p.grad = buf[o:o + p.numel()].view(p.shape)
        self.flat_grad = buf
        self._grad_views = None
        self._build_tables()

    def _ptr_of(self, p: Optional[torch.Tensor], grad: bool):
        if p is None:
            return None
        idx = self._index[id(p)]
        if grad:
            if not p.requires_grad:
                return None
            return self.flat_grad.data_ptr() + 4 * self.offsets[idx]
        return self.flat.data_ptr() + 4 * self.offsets[idx]

    def _build_tables(self):
        net = self.net
        self._index = {id(p): i for i, p in enumerate(self.params)}
        B = CONSTS

        def put(table_p, table_g, tensor):
            return self._ptr_of(tensor, False), self._ptr_of(tensor, True)

        def set2(arrP, arrG, i, tensor):
            arrP[i], arrG[i] = self._ptr_of(tensor, False), self._ptr_of(tensor, True)

        P, G = self.P, self.G
        conv, bn = net.conv1[0], net.conv1[2]
        for i, t in enumerate((conv.weight, conv.bias, bn.weight, bn.bias)):
            set2(P.stem, G.stem, i, t)
        for i in range(4):
            rw = getattr(net, f"rwattn{i + 1}", None)
            set2(P.table, G.table, i, rw.relative_position_bias_table if rw is not None else None)
        bi = 0
        le_mode = None
        for lname in LAYER_NAMES:
            for blk in _blocks_of(getattr(net, lname)):
                mlp, attn = blk.mlp, blk.attn
                lew = None
                mode = CONSTS["RL_LE_NONE"]
                if getattr(mlp, "local_enhence", False):
                    if mlp.use_partial:
                        lew, mode = mlp.leconv.partial_conv3.weight, CONSTS["RL_LE_PARTIAL"]
                    else:
                        lew, mode = mlp.leconv.weight, CONSTS["RL_LE_DEPTHWISE"]
                if le_mode is None:
                    le_mode = mode
                elif le_mode != mode:
                    raise _lib.RalenetError("mixed local-enhancement modes across blocks are not supported")
                ts = {
                    B["RL_BLK_WQ"]: attn.qkv_proj.to_q.weight, B["RL_BLK_BQ"]: attn.qkv_proj.to_q.bias,
                    B["RL_BLK_WKV"]: attn.qkv_proj.to_kv.weight, B["RL_BLK_BKV"]: attn.qkv_proj.to_kv.bias,
                    B["RL_BLK_WP"]: attn.proj.weight, B["RL_BLK_BP"]: attn.proj.bias,
                    B["RL_BLK_LN1W"]: blk.norm1.weight, B["RL_BLK_LN1B"]: blk.norm1.bias,
                    B["RL_BLK_LN2W"]: blk.norm2.weight, B["RL_BLK_LN2B"]: blk.norm2.bias,
                    B["RL_BLK_W1"]: mlp.fc1.weight, B["RL_BLK_B1"]: mlp.fc1.bias,
                    B["RL_BLK_W2"]: mlp.fc2.weight, B["RL_BLK_B2"]: mlp.fc2.bias, B["RL_BLK_LEW"]: lew,
                }
                for k, t in ts.items():
                    set2(P.blk[bi], G.blk[bi], k, t)
                bi += 1
        assert bi == CONSTS["RL_NBLOCKS"]
        self.le_mode = le_mode
        for j in range(4):
            pm, ps = getattr(net, f"pm{j + 1}"), getattr(net, f"ps{j + 1}")
            for i, t in enumerate((pm.reduction.weight, pm.norm.weight, pm.norm.bias)):
                set2(P.pm[j], G.pm[j], i, t)
            for i, t in enumerate((ps.reduction.weight, ps.norm.weight, ps.norm.bias)):
                set2(P.ps[j], G.ps[j], i, t)
        head = net.transconv[0]
        set2(P.head, G.head, 0, head.weight)
        set2(P.head, G.head, 1, head.bias)

    def refresh_requires_grad(self):
        """pointer tables encode requires_grad (frozen parameters get NULL gradient slots)."""
        sig = tuple(p.requires_grad for p in self.params)
        if getattr(self, "_rg_sig", None) != sig:
            self._build_tables()
            self._rg_sig = sig

    def attach_grads(self):
        """make every trainable Parameter's .grad a view of the flat gradient buffer.  A parameter whose .grad is
        None (optimizer.zero_grad(set_to_none=True), a newly unfrozen parameter) gets its slice zeroed; a foreign
        .grad tensor is folded into its slice; slices that are already aliased keep what they have accumulated.
        Returns True if anything had to be attached."""
        fresh = False
        base = self.flat_grad.data_ptr()
        todo = []
        for p, o in zip(self.params, self.offsets):
            if not p.requires_grad:
                continue
            g = p.grad
            if g is None or g.data_ptr() != base + 4 * o:
                todo.append((p, o, g))
        if not todo:
            return False
        fresh = True
        if self._grad_views is None:        # the views are built once (slicing 311 tensors per step costs ~1 ms)
            self._grad_views = {id(p): self.flat_grad[o:o + p.numel()].view(p.shape)
                                for p, o in zip(self.params, self.offsets)}
        views = self._grad_views
        n_train = sum(1 for p in self.params if p.requires_grad)
        if len(todo) == n_train and all(g is None for _, _, g in todo):
            self.flat_grad.zero_()          # the standard case after zero_grad(set_to_none=True): one memset
            for p, o, _ in todo:
                p.grad = views[id(p)]
            return fresh
        for p, o, g in todo:
            view = views[id(p)]
            if g is None:
                view.zero_()
            else:
                view.copy_(g)
            p.grad = view
        return fresh

    def cfg(self, B: int, L0: int, training: bool, save: bool, ws: torch.Tensor, flags: int = 0):
        net = self.net
        bn = net.conv1[2]
        if self.pe_L0 != L0 or self.pe is None or self.pe[0].device != self.flat.device:
            self.pe = [pos_table(L0 >> s, 8 << s, self.flat.device) for s in range(5)]
            self.pe_L0 = L0
        c = STRUCTS["rl_net_cfg"]()
        c.B, c.L0, c.le_mode, c.training, c.save, c.flags = B, L0, self.le_mode, int(training), int(save), flags
        for s in range(5):
            c.pe[s] = self.pe[s].data_ptr()
        c.running_mean, c.running_var = bn.running_mean.data_ptr(), bn.running_var.data_ptr()
        c.num_batches_tracked = bn.num_batches_tracked.data_ptr() if bn.num_batches_tracked is not None else None
        c.bn_stats = self.bn_stats.data_ptr()
        c.ws, c.ws_bytes = ws.data_ptr(), ws.numel()
        return c


# Per-GPU batches up to this many windows capture the training step on a HIGH-priority stream (see _capture_stream).
PRIO_MAX_BATCH = 768


def _capture_stream(batch: int):
    """stream the step graph is captured on.  Kernel nodes inherit the launch priority of their capture stream, and
    net.cu forks the weight-gradient GEMMs of the backward pass to a stream of the lowest priority.  While a launch of
    the data-gradient chain is at most two or three waves of CTAs (one window per CTA, 296 slots), ranking the chain above
    that branch lets its CTAs take freed SM slots first and the weight-gradient CTAs fill what is left: measured on one
    B200 (profiles/r2_v50_exp_prio*.txt) 1.910 -> 1.778 ms per step at 256 windows, 2.927 -> 2.798 at 384, 3.400 -> 3.313
    at 512, 4.887 -> 4.835 at 768.  With more waves the same ranking starves the branch until the chain has to wait for
    it (1024 windows: 6.06 -> 6.10 ms, 2048: 11.47 -> 11.96, 4096: 22.41 -> 23.19), so larger batches keep equal
    priorities (PRIO_MAX_BATCH).
    RALENET_MAIN_PRIO overrides (0 = lowest = torch's default, negative = higher)."""
    env = os.environ.get("RALENET_MAIN_PRIO")
    if env is not None and env != "":
        return torch.cuda.Stream(priority=int(env))
    if batch <= PRIO_MAX_BATCH:
        return torch.cuda.Stream(priority=torch.cuda.Stream.priority_range()[1])
    return None


def workspace_bytes(B: int, L0: int, save: bool, flags: int = 0) -> int:
    """bytes of the whole-network workspace; flags = RL_NET_DETERMINISTIC adds the partial slabs of the
    deterministic backward."""
    return int(_lib.load().ralenet_net_workspace_bytes_ex(B, L0, int(save), flags))


def _call(name, *args):
    _lib.check(getattr(_lib.load(), name)(*args))


class _WsLease:
    """a workspace buffer borrowed from the plan's pool; returned when the last reference (the autograd node of the
    forward that filled it) is released.  Keeps ralenet.forward from allocating a new 466 MB buffer per call."""
    __slots__ = ("buf", "pool")

    def __init__(self, buf, pool):
        self.buf, self.pool = buf, pool

    def __del__(self):
        try:
            if self.pool is not None and len(self.pool) < 4:
                self.pool.append(self.buf)
        except Exception:      # noqa: BLE001 -- interpreter shutdown
            pass


def _lease_ws(plan: NetPlan, nbytes: int, device) -> _WsLease:
    if torch.cuda.is_current_stream_capturing():
        # a captured forward keeps using its workspace at every replay, on whatever stream the graph is launched:
        # the buffer (from the graph's private pool) must never be handed to another forward
        return _WsLease(torch.empty(nbytes, device=device, dtype=torch.uint8), None)
    # one pool per (plan, stream): a returned buffer is only handed to work enqueued on the same stream, which
    # orders the reuse after the kernels that last touched it
    pool = plan.__dict__.setdefault("_ws_pools", {}).setdefault((str(device), _stream()), [])
    for i, b in enumerate(pool):
        if b.numel() == nbytes:
            return _WsLease(pool.pop(i), pool)
    del pool[:]                                   # another shape: drop the cached buffers
    return _WsLease(torch.empty(nbytes, device=device, dtype=torch.uint8), pool)


def _check_input(x):
    x = _chk(x, "x")
    if x.dim() != 3 or x.shape[1] != 2:
        raise _lib.RalenetError(f"ralenet expects (B, 2, L) windows (conv1 is Conv1d(2, 8, 3), "
                                f"model/transformer.py:571); got {tuple(x.shape)}")
    return x


def _forward_impl(plan: NetPlan, x, save: bool, flags: int = 0):
    B, _, L0 = x.shape
    plan.ensure(x.device)
    plan.refresh_requires_grad()
    training = plan.net.training
    lease = _lease_ws(plan, workspace_bytes(B, L0, save, flags), x.device)
    cfg = plan.cfg(B, L0, training, save, lease.buf, flags)
    out = torch.empty(B, 2, L0, device=x.device, dtype=torch.float32)
    st = ctypes.c_void_p(_stream())
    if training:
        _call("ralenet_net_fwd_stats", ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.c_void_p(x.data_ptr()), st)
        if plan.reduce_fn is not None:
            plan.reduce_fn(plan.bn_stats[:17])
    _call("ralenet_net_fwd", ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.c_void_p(x.data_ptr()),
          ctypes.c_void_p(out.data_ptr()), st)
    return out, lease, training


# inference precisions of a forward without an autograd node (_RalenetBase.inference_precision) -> rl_net_cfg.flags
INFERENCE_PRECISIONS = {"fp32": 0, "tf32": CONSTS["RL_NET_TF32"]}


def check_precision(value) -> str:
    if not isinstance(value, str) or value not in INFERENCE_PRECISIONS:
        raise ValueError(f"inference precision must be one of {sorted(INFERENCE_PRECISIONS)}, got {value!r}")
    return value


def forward_no_grad(plan: NetPlan, x):
    """ralenet.forward without an autograd node (torch.no_grad() / nothing requires grad): nothing is saved, the
    workspace is the 7-tensors-per-window ping/pong form (`save = 0` of net.cu::carve).  Runs in the module's
    inference_precision ("tf32": RL_NET_TF32, single-pass TF32 block GEMMs)."""
    x = _check_input(x)
    flags = INFERENCE_PRECISIONS[check_precision(plan.net.inference_precision)]
    out, lease, _ = _forward_impl(plan, x, save=False, flags=flags)
    plan.last_ws_bytes = lease.buf.numel()
    return out


class RalenetFn(torch.autograd.Function):
    """ralenet.forward (model/transformer.py:621-667) as one autograd node.
    `anchor` is a dummy leaf that requires grad whenever any parameter does, so that autograd calls
    backward even when x itself needs no gradient; parameter gradients are accumulated into the
    Parameters' .grad views of the flat gradient buffer as a side effect.  (Grad mode is decided by the caller,
    _RalenetBase.forward: inside Function.forward it is always off.)"""

    @staticmethod
    def forward(ctx, x, anchor, plan: NetPlan):
        x = _check_input(x)
        B, _, L0 = x.shape
        save = bool(ctx.needs_input_grad[0] or ctx.needs_input_grad[1])
        # torch.use_deterministic_algorithms(True) at forward time selects the deterministic backward; the
        # workspace is sized for it here and the backward follows this choice
        flags = _lib.RL_NET_DETERMINISTIC if save and torch.are_deterministic_algorithms_enabled() else 0
        out, lease, training = _forward_impl(plan, x, save, flags)
        plan.last_ws_bytes = lease.buf.numel()
        if save:
            ctx.plan, ctx.ws, ctx.shape, ctx.training, ctx.flags = plan, lease, (B, L0), training, flags
            # BN stats of THIS forward are needed by its backward; keep a private copy
            ctx.bn_stats = plan.bn_stats.clone() if training else None
            ctx.save_for_backward(x)
        return out

    @staticmethod
    def backward(ctx, dout):
        plan: NetPlan = ctx.plan
        (x,) = ctx.saved_tensors
        B, L0 = ctx.shape
        dout = _chk(dout, "grad_output")
        if not ctx.flags:
            _lib.deterministic_guard("ralenet backward of a forward run without torch.use_deterministic_algorithms(True)")
        plan.ensure(x.device)
        plan.attach_grads()
        if ctx.bn_stats is not None:
            plan.bn_stats[:17].copy_(ctx.bn_stats[:17])
        # the saved activations are only read by the backward kernels (their scratch is a separate part of the
        # workspace), so the node can be differentiated again under retain_graph=True: the lease lives as long as ctx
        cfg = plan.cfg(B, L0, ctx.training, True, ctx.ws.buf, ctx.flags)
        st = ctypes.c_void_p(_stream())
        _call("ralenet_net_bwd", ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.byref(plan.G),
              ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(dout.data_ptr()), st)
        if ctx.training and plan.reduce_fn is not None:
            plan.reduce_fn(plan.bn_stats[32:48])
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        _call("ralenet_net_bwd_stem", ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.byref(plan.G),
              ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(dx.data_ptr() if dx is not None else None), st)
        return dx, None, None


class _HostPipeline:
    """Host side of a software-pipelined training loop, shared by FusedTrainer and FineTuneTrainer:
    prefetch_host() copies the NEXT batch host -> device on a copy stream under the running step, step_host() picks the
    staged copy up, read_async() brings a step result back without stalling the enqueue of the following steps.
    The trainer provides _host_static(shape) -> (x, target) static device buffers."""
    _stage = None                     # staging pair, copy stream, events
    _staged_key = None
    _loss_slots = None                # pinned result slots

    def prefetch_host(self, hx: torch.Tensor, ht: torch.Tensor) -> None:
        """input-pipeline prefetch (what a DataLoader with pin_memory + non_blocking copies does): start the H2D copy of
        the NEXT batch from (pinned) HOST tensors into a staging pair on a copy stream, so that it runs under the step
        that is executing; the next step_host() called with the same two tensors takes the staged copy (a device to
        device copy) instead of copying from the host.  The batch is captured when this is called."""
        sx, st_ = self._host_static(hx.shape)
        dev = sx.device
        if self._stage is None or self._stage[0].shape != sx.shape:
            self._stage = (torch.empty_like(sx), torch.empty_like(st_))
            self._copy_stream = torch.cuda.Stream(dev)
            self._stage_ready, self._stage_free = torch.cuda.Event(), torch.cuda.Event()
            self._stage_free.record(torch.cuda.current_stream(dev))
        cs = self._copy_stream
        cs.wait_event(self._stage_free)               # the previous staged batch has been moved to the static buffers
        with torch.cuda.stream(cs):
            self._stage[0].copy_(hx, non_blocking=True)
            self._stage[1].copy_(ht, non_blocking=True)
            self._stage_ready.record(cs)
        self._staged_key = (hx.data_ptr(), ht.data_ptr(), tuple(hx.shape))

    def _load_host_batch(self, hx: torch.Tensor, ht: torch.Tensor):
        """static device buffers <- the copy prefetch_host() staged for these tensors, else the host tensors."""
        sx, st_ = self._host_static(hx.shape)
        if self._staged_key == (hx.data_ptr(), ht.data_ptr(), tuple(hx.shape)):
            main = torch.cuda.current_stream(sx.device)
            main.wait_event(self._stage_ready)
            sx.copy_(self._stage[0], non_blocking=True)
            st_.copy_(self._stage[1], non_blocking=True)
            self._stage_free.record(main)
            self._staged_key = None
        else:
            sx.copy_(hx, non_blocking=True)
            st_.copy_(ht, non_blocking=True)
        return sx, st_

    def read_async(self, dev_scalar: torch.Tensor):
        """start the device -> host copy of a step result (e.g. the loss tensor step_host() returned -- with use_graph
        that is a static buffer the next replay overwrites) into a pinned slot and return a callable that waits for
        it and gives the Python float.  Lets a loop enqueue steps i + 1, i + 2 before it reads the loss of step i, so
        the GPU never idles on the host round trip (at most 3 results may be outstanding)."""
        if self._loss_slots is None:
            self._loss_slots = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(4)]
            self._loss_events = [torch.cuda.Event() for _ in range(4)]
            self._loss_i = 0
        k = self._loss_i
        self._loss_i = (k + 1) % 4
        slot, ev = self._loss_slots[k], self._loss_events[k]
        slot.copy_(dev_scalar.reshape(1), non_blocking=True)
        ev.record(torch.cuda.current_stream(dev_scalar.device))

        def result() -> float:
            ev.synchronize()
            return float(slot[0])
        return result


class FusedTrainer(_HostPipeline):
    """The fast training path around the same kernels: fused MSE + metrics, flat Adam, and the whole
    step (fwd + loss + bwd + [grad all-reduce] + Adam) optionally replayed from a CUDA graph.

    Semantics = denoise_train.py:51-57 (zero_grad; model(data); F.mse_loss; backward; Adam lr 1e-3).
    Under torch.distributed the batch is sharded across ranks: BatchNorm statistics are all-reduced
    (SyncBN-equivalent, so the result equals the single-process step on the global batch) and the flat
    gradient buffer is all-reduced once (sum) in front of Adam.

    deterministic: True = bit-reproducible steps on one GPU (gradients, BatchNorm sums, loss, Adam trajectory; the
    backward writes partial slabs that are reduced in a fixed order, RL_NET_DETERMINISTIC); None = follow
    torch.are_deterministic_algorithms_enabled() at construction.  Not available with more than one rank.
    """

    def __init__(self, net: nn.Module, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 process_group=None, use_graph: bool = False, graph_collectives: Optional[bool] = None,
                 loss_weight: Optional[torch.Tensor] = None, deterministic: Optional[bool] = None):
        from . import ops
        self.ops = ops
        self.net = net
        # optional R-wave-weighted reconstruction loss (north-star extension; the reference's loss is plain MSE,
        # SURVEY F4): loss = mean(w * (pred - target)^2), w over the flattened (lead, sample) axis; None = F.mse_loss
        self.loss_weight = loss_weight
        self.plan: NetPlan = net._plan
        self.lr, self.betas, self.eps = lr, betas, eps
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        if self.world > 1:
            if deterministic:
                raise _lib.RalenetError("FusedTrainer(deterministic=True) is single-GPU only: the order of the "
                                        "multi-rank gradient exchange is not fixed")
            if deterministic is None:
                _lib.deterministic_guard("FusedTrainer with more than one rank")
            deterministic = False
        elif deterministic is None:
            deterministic = torch.are_deterministic_algorithms_enabled()
        self.deterministic = bool(deterministic)
        self.net_flags = _lib.RL_NET_DETERMINISTIC if self.deterministic else 0
        self.use_graph = use_graph
        # capture the NCCL all-reduces inside the step's CUDA graph (default; RALENET_GRAPH_NCCL=0 keeps them outside)
        self.graph_collectives = (os.environ.get("RALENET_GRAPH_NCCL", "1") != "0") if graph_collectives is None \
            else bool(graph_collectives)
        self.graph = None
        self.m = self.v = self.step_dev = None
        self._static = None
        # exchange steps: hand-written kernels over symmetric (peer / multicast) memory by default (comm.cu);
        # RALENET_COMM=nccl keeps the three torch.distributed all-reduces (the round-1 path, kept for A/B)
        self.comm = None
        self.comm_mode = os.environ.get("RALENET_COMM", "symm")
        self._synth = None            # synth_device.DeviceSynth feeding the step (step_synth)

    def _allreduce(self, t: torch.Tensor):
        torch.distributed.all_reduce(t, group=self.pg)

    def _setup(self, x: torch.Tensor):
        plan = self.plan
        _lib.check_device(x.device.index if x.device.index is not None else torch.cuda.current_device())
        plan.ensure(x.device)
        plan.refresh_requires_grad()
        if self.m is None or self.m.numel() != plan.flat.numel() or self.m.device != x.device:
            self.m = torch.zeros_like(plan.flat)
            self.v = torch.zeros_like(plan.flat)
            self.step_dev = torch.zeros(1, device=x.device, dtype=torch.int32)
        plan.reduce_fn = self._allreduce if self.world > 1 else None
        if self.world > 1 and self.comm_mode != "nccl":
            comm = getattr(plan, "_comm", None)
            if comm is None or comm.n != plan.n_flat or comm.device != x.device:
                from .comm import SymmComm
                try:
                    comm = SymmComm.create(plan.n_flat, x.device, self.pg)
                except Exception as e:      # noqa: BLE001 -- no symmetric memory on this system: NCCL all-reduces
                    import warnings
                    warnings.warn(f"FusedTrainer: symmetric-memory exchange unavailable ({type(e).__name__}: {e}); "
                                  "using NCCL all-reduces")
                    comm, self.comm_mode = None, "nccl"
                plan._comm = comm
            self.comm = comm
            if comm is not None:
                plan.rebind_grad(comm.grad)
        # frozen parameters must not move: mask = requires_grad
        if any(not p.requires_grad for p in plan.params):
            mask = torch.zeros_like(plan.flat)
            for p, o in zip(plan.params, plan.offsets):
                if p.requires_grad:
                    mask[o:o + p.numel()] = 1
            self.mask = mask
        else:
            self.mask = None

    def _pieces(self, x, target):
        """the step as an ordered list of ("compute" | "collective", fn) pieces; collectives only when world > 1.
        Results are left in self._res = (loss, rmse, snr, out)."""
        plan, ops = self.plan, self.ops
        B, _, L0 = x.shape
        ws, out = self._ws, self._out
        xp = ctypes.c_void_p(x.data_ptr())

        def cfg():
            return plan.cfg(B, L0, True, True, ws, self.net_flags)

        def st():
            return ctypes.c_void_p(_stream())

        def seg_a():
            self.net.train()
            if self._synth is not None:       # draw this step's batch on the device (batch index = Adam step counter)
                self._synth.fill(x, target, self.step_dev)
            plan.flat_grad.zero_()
            _call("ralenet_net_fwd_stats", ctypes.byref(cfg()), ctypes.byref(plan.P), xp, st())

        def seg_b():
            c = cfg()
            _call("ralenet_net_fwd", ctypes.byref(c), ctypes.byref(plan.P), xp, ctypes.c_void_p(out.data_ptr()), st())
            loss, dout, rmse, snr = ops.mse_loss_metrics(out, target, True, 1.0, out.numel() * self.world,
                                                         weight=self.loss_weight, partials=self._loss_partials)
            _call("ralenet_net_bwd", ctypes.byref(c), ctypes.byref(plan.P), ctypes.byref(plan.G), xp,
                  ctypes.c_void_p(dout.data_ptr()), st())
            self._res = (loss, rmse, snr, out)
            self._dout = dout

        def seg_c():
            _call("ralenet_net_bwd_stem", ctypes.byref(cfg()), ctypes.byref(plan.P), ctypes.byref(plan.G), xp,
                  ctypes.c_void_p(None), st())

        def seg_d():
            if self.mask is not None:
                plan.flat_grad.mul_(self.mask)
            ops.adam_flat(plan.flat, plan.flat_grad, self.m, self.v, self.step_dev, self.lr, self.betas, self.eps, 1.0)

        if self.world == 1:
            return [("compute", lambda: (seg_a(), seg_b(), seg_c(), seg_d()))]

        if self.comm is not None:
            comm = self.comm

            def fused():
                # the whole data-parallel step as plain kernel launches: no NCCL node, one CUDA graph
                seg_a()
                comm.exchange(0, plan.bn_stats[:17])
                seg_b()
                plan.bn_stats[48:49].copy_(self._res[0])      # the loss rides along with the 16 backward sums
                comm.exchange(1, plan.bn_stats[32:49])
                self._res[0].copy_(plan.bn_stats[48:49])
                seg_c()
                if self.mask is not None:
                    plan.flat_grad.mul_(self.mask)
                comm.allreduce_adam(plan.flat, self.m, self.v, self.step_dev, self.lr, self.betas, self.eps, 1.0)
            return [("compute", fused)]

        def ar_bwd_stats():
            # the 16 BN backward sums and the loss share one all-reduce (slot 48 of bn_stats is free)
            plan.bn_stats[48:49].copy_(self._res[0])
            self._allreduce(plan.bn_stats[32:49])
            self._res[0].copy_(plan.bn_stats[48:49])

        return [("compute", seg_a), ("collective", lambda: self._allreduce(plan.bn_stats[:17])),
                ("compute", seg_b), ("collective", ar_bwd_stats),
                ("compute", seg_c),
                ("collective", lambda: self._allreduce(plan.flat_grad)),
                ("compute", seg_d)]

    def _step_impl(self, x, target):
        for _, fn in self._pieces(x, target):
            fn()
        return self._res

    def _prepare(self, shape, device):
        if self._static is not None and tuple(self._static[0].shape) == tuple(shape):
            return
        B, _, L0 = shape
        probe = torch.empty(0, device=device)
        self._setup(probe)
        self._ws = torch.empty(workspace_bytes(B, L0, True, self.net_flags), device=device, dtype=torch.uint8)
        self._loss_partials = torch.empty(B, device=device, dtype=torch.float32) if self.deterministic else None
        self._out = torch.empty(B, 2, L0, device=device, dtype=torch.float32)
        self._static = (torch.empty(shape, device=device, dtype=torch.float32),
                        torch.empty(shape, device=device, dtype=torch.float32))
        self.graph = None

    def _replay(self):
        """graph mode: every compute piece is captured once into its own CUDA graph (one shared memory pool);
        NCCL collectives stay outside the graphs and are enqueued between the replays."""
        sx, st_ = self._static
        if self.graph is None:
            # warm up on a side stream (also initialises NCCL communicators), then capture
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            bn = self.net.conv1[2]
            snap = (self.plan.flat.clone(), self.m.clone(), self.v.clone(), self.step_dev.clone(),
                    bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone())
            with torch.cuda.stream(s):
                self._step_impl(sx, st_)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            # undo the warm-up step so that capture + replay applies exactly one update per call
            self.plan.flat.copy_(snap[0]); self.m.copy_(snap[1]); self.v.copy_(snap[2]); self.step_dev.copy_(snap[3])
            bn.running_mean.copy_(snap[4]); bn.running_var.copy_(snap[5]); bn.num_batches_tracked.copy_(snap[6])
            plan = None
            if self.world > 1 and self.graph_collectives:
                # one graph for the whole step, NCCL all-reduces captured as graph nodes (no host round trip and
                # no launch gap between the segments); falls back to the segmented form if capture is refused
                try:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=_capture_stream(sx.shape[0]), capture_error_mode="thread_local"):
                        for _, fn in self._pieces(sx, st_):
                            fn()
                    plan = [(g, None)]
                except Exception as e:      # noqa: BLE001 -- any capture failure means "use the segmented form"
                    import warnings
                    warnings.warn(f"FusedTrainer: NCCL graph capture failed ({e}); using segmented graphs")
                    torch.cuda.synchronize()
                    plan = None
            if plan is None:
                plan = []
                pool = None
                for kind, fn in self._pieces(sx, st_):
                    if kind == "collective":
                        plan.append((None, fn))
                        continue
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, pool=pool, stream=_capture_stream(sx.shape[0]),
                                          capture_error_mode="thread_local"):
                        fn()
                    pool = g.pool()
                    plan.append((g, None))
            self.graph = plan
            self._graph_out = self._res
            # capture does not execute: the replay below performs the step
        for g, fn in self.graph:
            if g is not None:
                g.replay()
            else:
                fn()
        return self._graph_out

    def close(self):
        """drop the captured graphs (call before destroying the process group)."""
        self.graph = None
        self._graph_out = None

    def step(self, x: torch.Tensor, target: torch.Tensor):
        """one training step on DEVICE tensors x, target of shape (B, 2, L).  Returns (loss[1], rmse[B], snr[B],
        out) as device tensors (no host sync)."""
        x, target = _chk(x, "x"), _chk(target, "target")
        self._prepare(x.shape, x.device)
        self._set_synth(None)
        if not self.use_graph:
            return self._step_impl(x, target)
        sx, st_ = self._static
        sx.copy_(x, non_blocking=True)
        st_.copy_(target, non_blocking=True)
        return self._replay()

    def _set_synth(self, synth):
        if self._synth is not synth:
            self._synth = synth
            self.graph = None             # the captured step changes

    def step_synth(self, synth):
        """one training step on a batch drawn ON THE DEVICE by `synth` (synth_device.DeviceSynth for synthetic windows,
        record_sampler.RecordSampler for windows of real record banks; anything with B, leads, L, device and
        fill(noisy, clean, counter)): no host traffic at all; with use_graph the generator is part of the step's CUDA
        graph and every replay sees new windows.  Returns (loss[1], rmse[B], snr[B], out) like step()."""
        self._prepare((synth.B, synth.leads, synth.L), synth.device)
        self._set_synth(synth)
        sx, st_ = self._static
        return self._replay() if self.use_graph else self._step_impl(sx, st_)

    def _host_static(self, shape):
        self._prepare(shape, next(self.net.parameters()).device)
        return self._static

    def step_host(self, hx: torch.Tensor, ht: torch.Tensor) -> torch.Tensor:
        """one training step from (pinned) HOST tensors: async H2D of the batch into the static device buffers (or the
        copy prefetch_host() staged for these tensors), then the step; returns the device loss tensor (the caller's
        .item() -- or read_async() -- is the D2H read)."""
        self._set_synth(None)
        sx, st_ = self._load_host_batch(hx, ht)
        return (self._replay() if self.use_graph else self._step_impl(sx, st_))[0]


class FineTuneTrainer(_HostPipeline):
    """The fast path of the 12-lead fine-tuning step (Transfer_learning.py:71-82 driving denoise_train.py:51-57):
    `newrale` = Conv1d(12->6,k13) -> Conv1d(6->2,k13) -> frozen RA-LENet core -> Conv1d(2->6,k13) -> Conv1d(6->12,k13)
    (model/ralenet_12leads.py:680-709), MSE, Adam(lr 1e-3) on the 2,210 parameters of the four convolutions.
    Same kernels as the drop-in module path (ops.Conv1dFn, RalenetFn), but enqueued straight through the C ABI on
    pre-allocated buffers -- no autograd graph, no per-tensor optimizer, one flat Adam -- so the whole step
    (forward, loss + metrics, data gradients through the frozen core, conv weight gradients, Adam) replays from ONE
    CUDA graph.  The core stays in whatever mode `model.rale.training` says (model.train() puts its BatchNorm in
    batch-statistics mode and updates its running statistics, exactly like the reference's frozen core).

    deterministic: True = bit-reproducible steps (loss, gradients, BatchNorm sums, Adam trajectory): the frozen core
    runs its RL_NET_DETERMINISTIC backward, the loss is summed in window order and the four convolutions write their
    weight gradients to per-window partial slabs reduced in window order (ralenet_conv1d_bwd_det); None = follow
    torch.are_deterministic_algorithms_enabled() at construction."""

    def __init__(self, model: nn.Module, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 use_graph: bool = False, deterministic: Optional[bool] = None):
        from . import ops
        self.ops, self.model, self.core = ops, model, model.rale
        self.lr, self.betas, self.eps, self.use_graph = lr, betas, eps, use_graph
        if deterministic is None:
            deterministic = torch.are_deterministic_algorithms_enabled()
        self.deterministic = bool(deterministic)
        self.net_flags = _lib.RL_NET_DETERMINISTIC if self.deterministic else 0
        self.convs = [model.conv1, model.conv2, model.conv3, model.conv4]
        self.slope = float(model.relu.negative_slope)
        self.flat = None
        self.graph = None
        self._shape = None
        self._source = None           # device batch source feeding the step (step_synth)

    def _setup(self, device):
        plan: NetPlan = self.core._plan
        plan.ensure(device)
        plan.refresh_requires_grad()
        ps = [p for c in self.convs for p in (c.weight, c.bias)]
        if self.flat is not None and all(p.data_ptr() == self.flat.data_ptr() + 4 * o for p, o in zip(ps, self.offs)):
            return
        offs, n = [], 0
        for p in ps:
            offs.append(n)
            n += (p.numel() + 3) // 4 * 4
        flat = torch.zeros(n, device=device, dtype=torch.float32)
        grad = torch.zeros_like(flat)
        with torch.no_grad():
            for p, o in zip(ps, offs):
                flat[o:o + p.numel()].copy_(p.detach().reshape(-1))
                p.data = flat[o:o + p.numel()].view(p.shape)
                p.grad = grad[o:o + p.numel()].view(p.shape)
        self.flat, self.flat_grad, self.offs, self.ps = flat, grad, offs, ps
        self.m, self.v = torch.zeros_like(flat), torch.zeros_like(flat)
        self.step_dev = torch.zeros(1, device=device, dtype=torch.int32)
        self.graph = None

    def _prepare(self, shape, device):
        self._setup(device)
        if self._shape == tuple(shape):
            return
        B, Cin, L = shape
        f = lambda c: torch.empty(B, c, L, device=device, dtype=torch.float32)
        self._x, self._t = f(Cin), f(Cin)
        self._a1, self._a2, self._r, self._a3, self._out = f(6), f(2), f(2), f(6), f(Cin)
        self._da3, self._dr, self._da2, self._da1 = f(6), f(2), f(2), f(6)
        self._ws = torch.empty(workspace_bytes(B, L, True, self.net_flags), device=device, dtype=torch.uint8)
        self._loss_partials = self._slabs = None
        if self.deterministic:
            self._loss_partials = torch.empty(B, device=device, dtype=torch.float32)
            # one slab per layer: no reuse between the four backward calls, whatever their launch order
            self._slabs = {}
            for c in self.convs:
                Co, Ci, K = c.weight.shape
                self._slabs[id(c)] = self.ops.conv1d_slab(B, Ci, Co, K, device)
        self._shape = tuple(shape)
        self.graph = None

    def _conv_fwd(self, x, conv, y, act):
        Co, Ci, K = conv.weight.shape
        a = _lib.STRUCTS["rl_conv_fwd_args"]()
        a.B, a.L, a.Cin, a.Cout, a.K, a.act, a.slope = x.shape[0], x.shape[2], Ci, Co, K, int(act), self.slope
        a.x, a.w, a.b, a.y = x.data_ptr(), conv.weight.data_ptr(), conv.bias.data_ptr(), y.data_ptr()
        _lib.call("ralenet_conv1d_fwd", a, _stream())

    def _conv_bwd(self, dy, x, conv, dx, act):
        Co, Ci, K = conv.weight.shape
        a = _lib.STRUCTS["rl_conv_bwd_args"]()
        a.B, a.L, a.Cin, a.Cout, a.K, a.act, a.slope = x.shape[0], x.shape[2], Ci, Co, K, int(act), self.slope
        a.dy, a.x, a.w, a.b = dy.data_ptr(), x.data_ptr(), conv.weight.data_ptr(), conv.bias.data_ptr()
        a.dx = dx.data_ptr() if dx is not None else None
        a.d_w, a.d_b = conv.weight.grad.data_ptr(), conv.bias.grad.data_ptr()
        if self._slabs is not None:
            self.ops.conv1d_bwd_det(a, self._slabs[id(conv)])
        else:
            _lib.call("ralenet_conv1d_bwd", a, _stream())

    def _step_impl(self):
        plan: NetPlan = self.core._plan
        c1, c2, c3, c4 = self.convs
        B, _, L = self._x.shape
        training = self.core.training
        st = ctypes.c_void_p(_stream())
        cfg = plan.cfg(B, L, training, True, self._ws, self.net_flags)
        a2p, rp = ctypes.c_void_p(self._a2.data_ptr()), ctypes.c_void_p(self._r.data_ptr())
        if self._source is not None:      # draw this step's batch on the device (batch index = Adam step counter)
            self._source.fill(self._x, self._t, self.step_dev)
        self.flat_grad.zero_()
        self._conv_fwd(self._x, c1, self._a1, True)
        self._conv_fwd(self._a1, c2, self._a2, True)
        if training:
            _call("ralenet_net_fwd_stats", ctypes.byref(cfg), ctypes.byref(plan.P), a2p, st)
        _call("ralenet_net_fwd", ctypes.byref(cfg), ctypes.byref(plan.P), a2p, rp, st)
        self._conv_fwd(self._r, c3, self._a3, True)
        self._conv_fwd(self._a3, c4, self._out, False)
        loss, dout, rmse, snr = self.ops.mse_loss_metrics(self._out, self._t, partials=self._loss_partials)
        self._conv_bwd(dout, self._a3, c4, self._da3, False)
        self._conv_bwd(self._da3, self._r, c3, self._dr, True)
        _call("ralenet_net_bwd", ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.byref(plan.G), a2p,
              ctypes.c_void_p(self._dr.data_ptr()), st)
        _call("ralenet_net_bwd_stem", ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.byref(plan.G), a2p,
              ctypes.c_void_p(self._da2.data_ptr()), st)
        self._conv_bwd(self._da2, self._a1, c2, self._da1, True)
        self._conv_bwd(self._da1, self._x, c1, None, True)
        self.ops.adam_flat(self.flat, self.flat_grad, self.m, self.v, self.step_dev, self.lr, self.betas, self.eps, 1.0)
        self._res = (loss, rmse, snr, self._out)
        self._keep = dout
        return self._res

    def _run(self, source=None):
        if source is not self._source:
            self._source = source
            self.graph = None             # the captured step changes
        if not self.deterministic:
            _lib.deterministic_guard("FineTuneTrainer constructed with deterministic=False")
        if not self.use_graph:
            return self._step_impl()
        if self.graph is None:
            bn = self.core.conv1[2]
            snap = (self.flat.clone(), self.m.clone(), self.v.clone(), self.step_dev.clone(), bn.running_mean.clone(),
                    bn.running_var.clone(), bn.num_batches_tracked.clone())
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._step_impl()                         # warm-up (loads kernels, sizes the allocator pool)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.flat.copy_(snap[0]); self.m.copy_(snap[1]); self.v.copy_(snap[2]); self.step_dev.copy_(snap[3])
            bn.running_mean.copy_(snap[4]); bn.running_var.copy_(snap[5]); bn.num_batches_tracked.copy_(snap[6])
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._step_impl()
            self.graph, self._graph_out = g, self._res
        self.graph.replay()
        return self._graph_out

    def step(self, x: torch.Tensor, target: torch.Tensor):
        """one fine-tuning step on DEVICE tensors (B, 12, L).  Returns (loss[1], rmse[B], snr[B], out)."""
        x, target = _chk(x, "x"), _chk(target, "target")
        self._prepare(x.shape, x.device)
        self._x.copy_(x, non_blocking=True)
        self._t.copy_(target, non_blocking=True)
        return self._run()

    def step_synth(self, source):
        """one fine-tuning step on a batch drawn ON THE DEVICE by `source` (e.g. record_sampler.RecordSampler on a
        12-lead bank; anything with B, leads, L, device and fill(noisy, clean, counter)), the counterpart of
        FusedTrainer.step_synth: the batch index is the Adam step counter, and with use_graph the draw is part of the
        step's CUDA graph.  Returns (loss[1], rmse[B], snr[B], out) like step()."""
        cin = self.convs[0].weight.shape[1]
        if source.leads != cin:
            raise ValueError(f"FineTuneTrainer.step_synth: the source draws {source.leads} leads, the model takes {cin}")
        self._prepare((source.B, source.leads, source.L), source.device)
        return self._run(source)

    def _host_static(self, shape):
        self._prepare(shape, self.convs[0].weight.device)
        return self._x, self._t

    def step_host(self, hx: torch.Tensor, ht: torch.Tensor) -> torch.Tensor:
        """the same from pinned HOST tensors (async H2D inside, or the copy prefetch_host() staged for these tensors);
        returns the device loss tensor."""
        self._load_host_batch(hx, ht)
        return self._run()[0]

    def close(self):
        self.graph = None
        self._graph_out = None
