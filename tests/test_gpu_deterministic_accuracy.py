"""Deterministic mode (RL_NET_DETERMINISTIC) against the fp64 oracle, element by element, on a poisoned workspace.

The deterministic backward writes every cross-CTA weight-gradient contribution into its own slot of a partial slab in
the workspace and grad_reduce_kernel (det.cu) sums the slots.  A wrong slot count or index gives the same wrong bits on
every run, so bit-identity between runs cannot see it, and a slot that is summed but never written reads whatever the
allocator left there.  Here every workspace is first filled with a byte pattern: 0xFF (NaN, caught wherever a stale
value is added or multiplied) or 0x7E (finite, ~8.5e37, caught where an fmaxf-style reduction would drop a NaN).

  * the drop-in backward of every kernel family and mode against the fp64 oracle (output, dx, every parameter
    gradient, BatchNorm running statistics) at batch edges the oracle can afford;
  * a sweep of the batch sizes at which the token-slice counts of the weight-gradient GEMMs change regime: poisoned
    and unpoisoned deterministic runs are bit-identical, and equal the atomic path up to summation order;
  * one FusedTrainer step (loss, metrics, gradients, BatchNorm statistics, Adam update) against the oracle.

The worst measured error of every comparison goes to $RALENET_PARITY_DIR/parity_det.json when that variable is set.
"""
import ctypes
import json
import math
import os
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import ralenet_oracle as O
from tests.common import rel_rms_err, switches
from tests.test_gpu_deterministic import _equal, _inputs, torch_deterministic

pytestmark = pytest.mark.gpu
RTOL = 1e-3
CROSS_RTOL = 5e-5          # deterministic vs atomic weight gradients: the same sums in another order
FAMILIES = ["default", "reg2", "mma"]
POISON = {"nan": 0xFF, "finite": 0x7E}
REPORT = {}
_ORACLE = {}


def _record(name, err):
    """keep the worst error per name; with RALENET_PARITY_DIR set, also write them to <dir>/parity_det.json."""
    REPORT[name] = max(float(err), REPORT.get(name, 0.0))
    out_dir = os.environ.get("RALENET_PARITY_DIR")
    if not out_dir:
        return
    try:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "parity_det.json"), "w") as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)
    except OSError:
        pass


# ------------------------------------------------------------------------------------------------------------------
# models, inputs and the cached fp64 oracle

# case: (variant, le, L0, depthwise local enhancement)
CASES = {"rw_le": ("rw", 1, 256, False), "rw_mlp": ("rw", 0, 256, False), "rw_dw": ("rw", 1, 256, True),
         "nra512": ("nra", 1, 512, False)}


def _model(case):
    from tests.test_gpu_inference_precision import _model as build
    variant, le, _, dw = CASES[case]
    return build(variant, le, 2023, depthwise=dw).train()


def _batch(B, L0):
    from ecg_denoise_b200 import synth
    noisy, clean = synth.make_batch(B, 2, L0, seed=100 + B)
    return torch.from_numpy(noisy), torch.from_numpy(clean)


def _centre_weight(L0):
    centre = np.exp(-0.5 * ((np.arange(L0) - L0 // 2) / 12.0) ** 2)
    return torch.from_numpy(np.concatenate([1 + 4 * centre, 1 + 4 * centre])).float()


def _oracle(case, B):
    """fp64 forward + backward of the case's model on _batch(B, L0): plain MSE, and for rw_le also the centre-weighted
    loss of the FusedTrainer test.  Only the results are cached (the tape of 515 windows is ~10 GB of host memory)."""
    L0 = CASES[case][2]
    key = (case, B, L0)
    if key not in _ORACLE:
        m = _model(case)
        sd = {k: (v.detach().double().cpu() if v.dtype.is_floating_point else v.cpu())
              for k, v in m.state_dict().items()}
        x, t = _batch(B, L0)
        out, ctx, stats = O.ralenet_fwd(x.double(), sd, training=True)
        loss, dout = O.mse_loss_fwd_bwd(out, t.double())
        dx, grads = O.ralenet_bwd(dout, ctx, sd)
        r = dict(out=out.numpy(), loss=float(loss), dx=dx.numpy(), grads={k: v.numpy() for k, v in grads.items()},
                 rmean=stats[0].numpy(), rvar=stats[1].numpy(), nbt=int(sd["conv1.2.num_batches_tracked"]) + 1,
                 snr=O.SNR(t.double(), out).numpy(), rmse=O.RMSE(t.double(), out).numpy())
        if case == "rw_le":
            wl, wd = O.weighted_mse_loss_fwd_bwd(out, t.double(), _centre_weight(L0).double())
            r["wloss"], r["wgrads"] = float(wl), {k: v.numpy() for k, v in O.ralenet_bwd(wd, ctx, sd)[1].items()}
        del ctx
        _ORACLE[key] = r
    return _ORACLE[key]


def _check(name, got, ref, rtol=RTOL):
    got, ref = np.asarray(got, np.float64).reshape(-1), np.asarray(ref, np.float64).reshape(-1)
    assert got.size == ref.size, (name, got.size, ref.size)
    e = rel_rms_err(got, ref)
    _record(name, e)
    assert math.isfinite(e) and e <= rtol, f"{name}: rel err {e:.3e} > {rtol}"


def _check_grads(tag, m, flat_grad, grads, rtol_of=lambda n: RTOL):
    """every parameter gradient (slices of the flat gradient buffer) against the oracle; the key half of to_kv.bias
    has an exact gradient of 0 (softmax is invariant to a per-query shift of the logits): asserted to be ~0."""
    plan = m._plan
    g = flat_grad.double().cpu().numpy()
    names = [n for n, _ in m.named_parameters()]
    assert sorted(names) == sorted(grads), set(names) ^ set(grads)
    for (n, p), o in zip(m.named_parameters(), plan.offsets):
        got = g[o:o + p.numel()]
        _check(f"{tag}/grad/{n}", got, grads[n], rtol_of(n))
        if n.endswith("to_kv.bias"):
            C = p.numel() // 2
            assert np.linalg.norm(got[:C]) <= 1e-5 * np.linalg.norm(got[C:]) + 1e-12, n


def _check_bn(tag, m, ref):
    bn = m.conv1[2]
    assert np.allclose(bn.running_mean.cpu().numpy(), ref["rmean"], rtol=1e-4, atol=1e-6), tag
    assert np.allclose(bn.running_var.cpu().numpy(), ref["rvar"], rtol=1e-4, atol=1e-6), tag
    assert int(bn.num_batches_tracked.item()) == ref["nbt"], tag


# ------------------------------------------------------------------------------------------------------------------
# poisoned workspaces

@pytest.fixture
def poison(monkeypatch):
    """poison(pattern): from now on every workspace the drop-in forward leases (engine._lease_ws, also the pooled
    buffers it hands out again) is filled with the byte `pattern` first (None: left as allocated).  Returns a list
    that counts the poisoned leases."""
    from ecg_denoise_b200 import engine
    lease_ws = engine._lease_ws
    state = {"byte": None}
    hits = []

    def poisoned(plan, nbytes, device):
        lease = lease_ws(plan, nbytes, device)
        if state["byte"] is not None:
            lease.buf.fill_(state["byte"])
            hits.append(nbytes)
        return lease

    monkeypatch.setattr(engine, "_lease_ws", poisoned)

    def set_pattern(byte):
        state["byte"] = byte
        return hits
    return set_pattern


def _poison_trainer(tr, shape, device, byte):
    """FusedTrainer: allocate the step buffers now and fill the workspace and the loss partials with `byte`."""
    tr._prepare(shape, device)
    tr._ws.fill_(byte)
    if tr._loss_partials is not None:
        tr._loss_partials.fill_(byte)
    return tr._ws.data_ptr()


def test_poison_patterns_fill_the_leased_workspace(poison):
    """the hook fills what _lease_ws hands out (fresh and pooled buffers), and the two patterns decode as intended."""
    from ecg_denoise_b200 import _lib, engine
    m = _model("rw_le")
    x, _ = _inputs(3, 256)
    with torch_deterministic():
        hits = poison(POISON["finite"])
        m(x).sum().backward()
    assert hits == [engine.workspace_bytes(3, 256, True, _lib.RL_NET_DETERMINISTIC)]
    for byte in POISON.values():
        poison(byte)
        lease = engine._lease_ws(m._plan, 4096, x.device)
        assert bool((lease.buf == byte).all())
    as_f32 = lambda b: torch.full((4,), b, dtype=torch.uint8).view(torch.float32).item()
    assert math.isnan(as_f32(POISON["nan"]))
    assert as_f32(POISON["finite"]) == pytest.approx(8.45e37, rel=1e-2)


# ------------------------------------------------------------------------------------------------------------------
# 1. the drop-in backward against the fp64 oracle

ORACLE_CASES = [
    ("rw_le", 1),        # several GEMM groups have M < 64 tokens: the register and tcgen05 families decline them
    ("rw_le", 37),       # ragged batch, one split per 128 tokens in the SIMT patch GEMMs
    ("rw_le", 515),      # the 148-slice cap binds in the SIMT patch GEMMs and the C = 32 feed-forward group
    ("rw_mlp", 37),      # no local enhancement
    ("rw_dw", 37),       # depthwise local enhancement: per-window feed-forward kernels at every stage, 12 C lew slots
    ("rw_dw", 515),
    ("nra512", 1),       # 512-sample windows (L * C = 4096: the two-window kernels)
    ("nra512", 37),
]


@contextmanager
def _mode(det):
    """torch.use_deterministic_algorithms(det) at forward time selects the deterministic or the atomic backward."""
    if det:
        with torch_deterministic():
            yield
    else:
        assert not torch.are_deterministic_algorithms_enabled()
        yield


def _dropin(m, x, t, det):
    """drop-in forward + F.mse_loss + backward; returns (out, loss, dx, flat_grad)."""
    xg = x.clone().requires_grad_(True)
    with _mode(det):
        y = m(xg)
        loss = torch.nn.functional.mse_loss(y, t)
        loss.backward()
    torch.cuda.synchronize()
    return y.detach(), loss.detach().item(), xg.grad, m._plan.flat_grad


@pytest.mark.parametrize("det", [True, False], ids=["det", "atomic"])
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("case,B", ORACLE_CASES, ids=[f"{c}-B{b}" for c, b in ORACLE_CASES])
def test_dropin_backward_vs_oracle_on_poisoned_workspace(poison, case, B, family, det):
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.engine import workspace_bytes
    ref = _oracle(case, B)
    L0 = CASES[case][2]
    x, t = (v.cuda() for v in _batch(B, L0))
    tag = f"{case}/B{B}/{family}/{'det' if det else 'atomic'}"
    with switches(family):
        m = _model(case)
        hits = poison(POISON["nan"])
        y, loss, dx, flat_grad = _dropin(m, x, t, det)
    flags = _lib.RL_NET_DETERMINISTIC if det else 0
    assert hits == [workspace_bytes(B, L0, True, flags)]
    assert m._plan.last_ws_bytes == workspace_bytes(B, L0, True, flags)
    _check(f"{tag}/out", y.cpu(), ref["out"])
    assert abs(loss - ref["loss"]) <= 1e-4 * abs(ref["loss"]), (loss, ref["loss"])
    _check(f"{tag}/dx", dx.cpu(), ref["dx"])
    _check_grads(tag, m, flat_grad, ref["grads"])
    _check_bn(tag, m, ref)


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


@pytest.mark.parametrize("family", FAMILIES)
def test_each_family_launches_its_deterministic_gemms(family):
    """the switches select the GEMM family the oracle tests claim to cover, and the slabs are reduced."""
    x, t = _inputs(37, 256)
    with switches(family):
        m = _model("rw_le")
        names = {l.split("<")[0] for l in _labels(lambda: _dropin(m, x, t, True))}
    assert "grad_reduce_kernel" in names
    if family == "default":
        assert {"wgrad_reg_kernel", "wgrad_umma_kernel", "wgrad_kernel"} <= names, names
    elif family == "reg2":
        assert {"wgrad_reg_kernel", "wgrad_kernel"} <= names and "wgrad_umma_kernel" not in names, names
    else:
        assert {"wgrad_group_kernel", "wgrad_kernel"} <= names, names
        assert not names & {"wgrad_umma_kernel", "wgrad_reg_kernel"}, names


# ------------------------------------------------------------------------------------------------------------------
# 2. batch edges of the token-slice counts: poisoned == unpoisoned bit for bit, deterministic ~ atomic
#
# Token slices per weight-gradient GEMM (M = tokens of the group; caps: RL_DET_MAX_SPLIT = 148 slices in deterministic
# mode).  L0 = 256, stage s has C = 8 << s channels and L = 256 >> s tokens per window; a patch layer of width CN has
# M = B * 2048 / CN tokens.  The SIMT kernels (wgrad.cu, widths 8 and 16) take one slice per 128 tokens, the register
# tiles (wgrad_reg.cu) one per 64 * (8 / tiles per CTA) tokens, mma.sync groups (wgrad.cu) one per 128 tokens.
EDGES = {
    256: [
        1,      # pm3 / ps4 (M = 32 B) and every stage-3/4 group below 64 tokens: register and tcgen05 families decline
        2,      # pm3 / ps4 reach M = 64: register tiles take them; stage-3 groups (M = 64) still below tcgen05's 128
        3,      # stage-3 attention / feed-forward groups at M = 96: still mma.sync (default family)
        4,      # ... at M = 128: tcgen05 takes them
        7,      # stage-4 groups (M = 112) still mma.sync
        8,      # ... at M = 128: tcgen05
        74,     # ps1 (width 8, M = 256 B): 148 slices, exactly the cap
        75,     # ps1: 150 slices wanted, capped (120 after rounding the slice length)
        76,
        148,    # pm1 / ps2 (width 16, M = 128 B): 148 slices, exactly the cap
        149,    # pm1 / ps2: capped
        150,
        297,    # mma family: pm2 / ps3 group (width 32, M = 64 B) capped from here
        298,    # register tiles: C = 32 feed-forward group capped (and, under reg2, the C = 64 attention group)
        593,    # mma family: pm3 / ps4 group (width 64) capped
        596,    # register tiles: C = 32 attention group, pm3 / ps4 capped (reg2: also pm4)
        1191,   # register tiles: pm2 / ps3 (width 32, one slice per 512 tokens) at 148 slices
        1192,   # ... capped
        4096,   # every GEMM at the cap; ~8 GB of workspace
    ],
    512: [      # L * C = 4096: twice the tokens per window, every threshold at half the batch
        1,      # stage-3 groups at M = 64: tcgen05 declines
        2,      # ... at M = 128: tcgen05
        37,     # ps1: 148 slices
        38,     # ps1: capped
        74,     # pm1 / ps2: 148 slices
        75,     # pm1 / ps2: capped
        148,    # mma: pm2 / ps3 at the cap; register tiles: C = 32 feed-forward group at the cap
        149,    # ... capped
        255,
        298,    # register tiles: C = 32 attention group, pm3 / ps4 capped
        1024,
    ],
}
EDGE_CASES = [(L0, B) for L0, bs in EDGES.items() for B in bs]


def _dropin_sums(m, x, t, det):
    """drop-in backward (ops.mse_loss_metrics dout, as the deterministic tests use): (loss, dx, flat_grad, BN sums)."""
    from ecg_denoise_b200 import ops
    xg = x.clone().requires_grad_(True)
    with _mode(det):
        m._plan.flat_grad.zero_() if m._plan.flat_grad is not None else None
        y = m(xg)
        loss, dout, _, _ = ops.mse_loss_metrics(y.detach(), t)
        y.backward(dout)
    torch.cuda.synchronize()
    res = (loss.clone(), xg.grad.clone(), m._plan.flat_grad.clone(), m._plan.bn_stats[32:48].clone())
    del y, xg
    return res


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("L0,B", EDGE_CASES, ids=[f"L{l}-B{b}" for l, b in EDGE_CASES])
def test_batch_edges_poison_invariant_and_match_atomic(poison, L0, B, family):
    x, t = _inputs(B, L0, seed=B)
    with switches(family):
        m = _model("rw_le" if L0 == 256 else "nra512")
        hits = poison(None)
        ref = _dropin_sums(m, x, t, True)
        for name, byte in POISON.items():
            n0 = len(poison(byte))
            got = _dropin_sums(m, x, t, True)
            assert len(hits) == n0 + 1
            _equal(ref, got, f"L{L0}/B{B}/{family}: {name}-poisoned workspace")
        poison(POISON["nan"])
        atomic = _dropin_sums(m, x, t, False)
    tag = f"det_vs_atomic/L{L0}/B{B}/{family}"
    assert torch.isfinite(ref[2]).all() and torch.isfinite(ref[1]).all()
    _check(f"{tag}/loss", ref[0].cpu(), atomic[0].double().cpu(), CROSS_RTOL)
    _check(f"{tag}/dx", ref[1].cpu(), atomic[1].double().cpu(), CROSS_RTOL)
    _check(f"{tag}/bn_sums", ref[3].cpu(), atomic[3].double().cpu(), CROSS_RTOL)
    g, ga = ref[2].double().cpu().numpy(), atomic[2].double().cpu().numpy()
    worst = 0.0
    for (n, p), o in zip(m.named_parameters(), m._plan.offsets):
        e = rel_rms_err(g[o:o + p.numel()], ga[o:o + p.numel()])
        worst = max(worst, e)
        assert math.isfinite(e) and e <= CROSS_RTOL, f"{tag}/{n}: {e:.3e}"
    _record(f"{tag}/grad_worst", worst)
    _record("det_vs_atomic/worst", worst)
    del m, ref, atomic
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------
# 3. one deterministic FusedTrainer step against the oracle

@pytest.mark.parametrize("weighted", [False, True], ids=["mse", "weighted"])
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("B", [37, 515])
def test_fused_trainer_deterministic_step_vs_oracle(B, graph, weighted):
    from ecg_denoise_b200.engine import FusedTrainer
    ref = _oracle("rw_le", B)
    x, t = (v.cuda() for v in _batch(B, 256))
    m = _model("rw_le")
    w = _centre_weight(256).cuda() if weighted else None
    tr = FusedTrainer(m, lr=1e-3, use_graph=graph, deterministic=True, loss_weight=w)
    ws = _poison_trainer(tr, x.shape, x.device, POISON["nan"])
    assert tr._loss_partials is not None and tr._loss_partials.numel() == B
    flat0 = m._plan.flat.double().cpu()
    loss, rmse, snr, out = tr.step(x, t)
    torch.cuda.synchronize()
    assert tr._ws.data_ptr() == ws                  # the poisoned buffers are the ones the step used
    tag = f"fused/B{B}/{'graph' if graph else 'eager'}/{'weighted' if weighted else 'mse'}"
    ref_loss = ref["wloss"] if weighted else ref["loss"]
    _record(f"{tag}/loss", abs(loss.item() - ref_loss) / abs(ref_loss))
    assert abs(loss.item() - ref_loss) <= 1e-4 * abs(ref_loss), (loss.item(), ref_loss)
    _check(f"{tag}/out", out.cpu(), ref["out"])
    assert np.max(np.abs(snr.cpu().numpy() - ref["snr"])) < 0.01
    assert np.max(np.abs(20 * np.log10(rmse.cpu().numpy() / ref["rmse"]))) < 0.01
    # the query projection of the widest stage sits on a cancellation that the centre-weighted loss sharpens
    # (test_gpu_net.py::test_fused_trainer_weighted_loss_step): 2e-3 there
    rt = (lambda n: 2e-3 if n.endswith("to_q.weight") else RTOL) if weighted else (lambda n: RTOL)
    g = m._plan.flat_grad.clone()
    _check_grads(tag, m, g, ref["wgrads"] if weighted else ref["grads"], rt)
    _check_bn(tag, m, ref)
    # the parameters after the step are Adam's first step on the step's own gradient, computed in fp64
    p64, g64 = flat0.clone(), g.double().cpu()
    O.adam_step(p64, g64, torch.zeros_like(p64), torch.zeros_like(p64), 1, lr=1e-3)
    got = m._plan.flat.double().cpu().numpy()
    worst = 0.0
    for (n, p), o in zip(m.named_parameters(), m._plan.offsets):
        e = rel_rms_err(got[o:o + p.numel()], p64[o:o + p.numel()].numpy())
        worst = max(worst, e)
        assert e <= 1e-5, f"{tag}/adam/{n}: {e:.3e}"
    _record(f"{tag}/adam_params", worst)
    tr.close()
