"""TF32 inference precision (inference_precision = "tf32", RL_NET_TF32) on the GPU.

The reduced-precision gate of BASELINE.md section 3: |out - ref| <= 1e-2 * (|ref| + rms(ref)) against the fp64 oracle,
and per-record SNR / RMSE within 0.01 dB of the fp32 mode.  Every forward kernel family that a no-grad forward reaches
is covered: the fused narrow-stage block kernel, the one- and two-window attention kernels, the per-window
feed-forward kernel (all three local-enhancement modes, 512-sample windows) and the tcgen05 tile kernels."""
import ctypes
from contextlib import contextmanager

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import ralenet_oracle as O
from oracle import synth_weights as SW
from tests.common import CASES, rel_rms_err

pytestmark = pytest.mark.gpu
GATE = 1e-2
_ORACLE = {}


def _model(variant="rw", le=1, seed=2023, depthwise=False):
    from ecg_denoise_b200.model import raletransformer, transformer
    m = raletransformer.ralenet() if variant == "nra" else transformer.ralenet(high_level_enhence=bool(le))
    m.load_state_dict(SW.make_state_dict(variant, le, seed), strict=True)
    if depthwise:      # Mlp(use_partial=False): per-channel 3-tap FIRs on all 4C hidden channels (RL_LE_DEPTHWISE)
        g = torch.Generator().manual_seed(seed)
        for mod in list(m.modules()):
            if hasattr(mod, "leconv"):
                hc = mod.fc1.out_features
                mod.use_partial = False
                mod.leconv = nn.Conv1d(hc, hc, 3, padding=1, groups=hc, bias=False)
                with torch.no_grad():
                    mod.leconv.weight.copy_(torch.randn(hc, 1, 3, generator=g) * 0.5)
    return m.cuda().eval()


def _oracle(key, m, x):
    """fp64 eval-mode oracle output, cached per (model, batch) key."""
    if key not in _ORACLE:
        sd = {k: (v.detach().double().cpu() if v.dtype.is_floating_point else v.cpu())
              for k, v in m.state_dict().items()}
        _ORACLE[key] = O.ralenet_fwd(x.double().cpu(), sd, training=False)[0].numpy()
    return _ORACLE[key]


def _run(m, x, precision):
    m.inference_precision = precision
    try:
        with torch.no_grad():
            return m(x)
    finally:
        m.inference_precision = "fp32"


@contextmanager
def attn_umma(mode):
    from ecg_denoise_b200 import _lib
    prev = _lib.set_attn_umma(mode)
    try:
        yield
    finally:
        _lib.set_attn_umma(prev)


def _gate(name, got, ref):
    e = rel_rms_err(got.double().cpu().numpy(), ref)
    print(f"{name}: rel err {e:.3e}")
    assert np.isfinite(e) and e <= GATE, f"{name}: rel err {e:.3e} > {GATE}"
    return e


@pytest.mark.parametrize("tag", list(CASES))
def test_golden_cases_meet_the_reduced_precision_gate(golden, tag):
    variant, le, seed, xk, _ = CASES[tag]
    m = _model(variant, le, seed)
    x = torch.from_numpy(golden[xk]).cuda()
    with torch.no_grad():
        y_default = m(x)
    y32 = _run(m, x, "fp32")
    yt = _run(m, x, "tf32")
    assert torch.equal(y32, y_default)                 # precision="fp32" is the default path, bit for bit
    assert not torch.equal(yt, y32)                    # the single-pass kernels really ran
    _gate(f"{tag}/tf32", yt, golden[f"{tag}/eval_out64"])


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("B", [256, 515, 1024])
def test_every_attention_kernel_selection_and_batch(B, mode):
    """mode 0: one- and two-window attention kernels; 2: tcgen05 tile kernels; 1: the default selection.  515 leaves
    an odd window for the one-window kernel behind the two-window groups (B >= 512)."""
    m = _model("rw", 1, 11)
    x = torch.randn(B, 2, 256, generator=torch.Generator().manual_seed(B)).cuda()
    with attn_umma(mode):
        yt = _run(m, x, "tf32")
        y32 = _run(m, x, "fp32")
    assert not torch.equal(yt, y32)
    _gate(f"B{B}/attn_umma{mode}", yt, _oracle(("rw_le", B), m, x))


@pytest.mark.parametrize("le", ["none", "partial", "depthwise"])
def test_every_local_enhancement_mode(le):
    """depthwise runs the per-window feed-forward kernel at every stage (the tile kernels do not take it)."""
    m = _model("rw", 0 if le == "none" else 1, 12, depthwise=(le == "depthwise"))
    x = torch.randn(300, 2, 256, generator=torch.Generator().manual_seed(3)).cuda()
    yt = _run(m, x, "tf32")
    assert not torch.equal(yt, _run(m, x, "fp32"))
    _gate(f"le_{le}", yt, _oracle(("le", le), m, x))


def _profiled_labels(m, x, precision):
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.ops import _stream
    lib = _lib.load()
    n, stride = 4096, 48
    labels, ms = ctypes.create_string_buffer(n * stride), (ctypes.c_float * n)()
    m.inference_precision = precision
    try:
        _lib.check(lib.ralenet_profile_begin(ctypes.c_void_p(_stream())))
        with torch.no_grad():
            m(x)
        got = lib.ralenet_profile_end(labels, stride, ms, n)
    finally:
        m.inference_precision = "fp32"
    assert got > 0
    return [labels.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode() for i in range(got)]


def test_profiled_forward_labels_every_block_forward_tf32():
    m = _model("rw", 1, 2023)
    x = torch.randn(256, 2, 256, generator=torch.Generator().manual_seed(1)).cuda()
    fams = ("block_fwd_kernel", "attn_fwd", "ffn_fwd")
    for precision in ("tf32", "fp32"):
        labels = _profiled_labels(m, x, precision)
        blk = [l for l in labels if l.startswith(fams)]
        print(precision, blk)
        # 10 narrow-stage blocks (C <= 32) in one fused launch each, 8 wide-stage blocks (C = 64, 128) as an attention
        # and a feed-forward launch
        assert sum(l.startswith("block_fwd_kernel") for l in blk) == 10
        assert sum(l.startswith("attn_fwd") for l in blk) == 8
        assert sum(l.startswith("ffn_fwd") for l in blk) == 8
        tf32 = [l for l in blk if l.endswith(":tf32")]
        assert len(tf32) == (len(blk) if precision == "tf32" else 0)
        assert not any(l.endswith(":tf32") for l in labels if not l.startswith(fams))


def test_tf32_forward_is_repeatable():
    m = _model("rw", 1, 2023)
    x = torch.randn(515, 2, 256, generator=torch.Generator().manual_seed(2)).cuda()
    assert torch.equal(_run(m, x, "tf32"), _run(m, x, "tf32"))


def _records(R, leads, nwin, tail, seed):
    """SNR-mixed synthetic records: clean beat trains (synth.py) of nwin windows plus a ragged tail, noise at -4 dB."""
    from ecg_denoise_b200 import synth
    w = synth.clean_windows(R * (nwin + 1), leads, 256, seed).reshape(R, nwin + 1, leads, 256)
    clean = np.ascontiguousarray(w.transpose(0, 2, 1, 3).reshape(R, leads, (nwin + 1) * 256)[..., :nwin * 256 + tail])
    noisy = synth.add_noise(clean, "emb", -4.0, seed + 1)
    return torch.from_numpy(noisy).cuda(), torch.from_numpy(clean)


def _snr_rmse_close(clean, y32, yt):
    snr32, snrt = O.SNR(clean, y32.cpu()).numpy(), O.SNR(clean, yt.cpu()).numpy()
    r32, rt = O.RMSE(clean, y32.cpu()).numpy(), O.RMSE(clean, yt.cpu()).numpy()
    d_snr, d_rmse = np.abs(snrt - snr32), np.abs(20 * np.log10(rt / r32))
    print(f"SNR fp32 {snr32} tf32 {snrt}; max |dSNR| {d_snr.max():.2e} dB, max |dRMSE| {d_rmse.max():.2e} dB")
    assert d_snr.max() < 0.01 and d_rmse.max() < 0.01


def test_denoise_records_tf32_within_0p01_db():
    from ecg_denoise_b200 import inference
    m = _model("rw", 1, 2023)
    noisy, clean = _records(6, 2, 40, 100, 7)
    y32 = inference.denoise_records(m, noisy, batch=97, precision="fp32")
    yt = inference.denoise_records(m, noisy, batch=97, precision="tf32")
    assert m.inference_precision == "fp32"                     # restored
    assert torch.equal(y32, inference.denoise_records(m, noisy, batch=97))
    assert not torch.equal(yt, y32)
    _snr_rmse_close(clean, y32, yt)


def test_denoise_records_tf32_newrale_12_leads():
    from ecg_denoise_b200 import inference
    from ecg_denoise_b200.model import ralenet_12leads as TW
    m = TW.newrale(TW.ralenet(high_level_enhence=True))
    m.load_state_dict(SW.make_newrale_state_dict(2023), strict=True)
    m = m.cuda()
    noisy, clean = _records(3, 12, 24, 0, 9)
    m.rale.inference_precision = "tf32"                        # precision="fp32" overrides it for the call only
    y32 = inference.denoise_records(m, noisy, batch=50, precision="fp32")
    assert m.rale.inference_precision == "tf32"
    m.rale.inference_precision = "fp32"
    yt = inference.denoise_records(m, noisy, batch=50, precision="tf32")
    assert m.rale.inference_precision == "fp32"
    assert not torch.equal(yt, y32)
    _snr_rmse_close(clean, y32, yt)


def _recorded_step(m, x):
    """forward recorded for a backward, and the backward, in deterministic mode (bit-reproducible gradients)"""
    state = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True)
    try:
        m.zero_grad(set_to_none=False)
        xg = x.clone().requires_grad_(True)
        y = m(xg)
        y.square().sum().backward()
        return y.detach(), xg.grad, {n: p.grad.clone() for n, p in m.named_parameters()}
    finally:
        torch.use_deterministic_algorithms(state[0], warn_only=state[1])


def test_recorded_forward_stays_fp32_and_backward_works():
    m = _model("rw", 1, 2023)
    x = torch.randn(64, 2, 256, generator=torch.Generator().manual_seed(4)).cuda()
    y32, dx32, g32 = _recorded_step(m, x)
    m.inference_precision = "tf32"
    yt, dxt, gt = _recorded_step(m, x)
    assert torch.equal(yt, y32)
    assert torch.isfinite(dxt).all() and torch.equal(dxt, dx32)
    for n in g32:
        assert torch.equal(gt[n], g32[n]), n
    with torch.no_grad():
        assert not torch.equal(m(x), y32)                      # the attribute is set: no-grad forwards use it


# -- C ABI rejections -----------------------------------------------------------------------------------------
def _f(n):
    return torch.zeros(n, device="cuda")


def _attn_args(flags, save):
    from ecg_denoise_b200 import _lib
    a = _lib.STRUCTS["rl_attn_fwd_args"]()
    a.B, a.L, a.C, a.H, a.W, a.c0, a.flags = 1, 256, 8, 2, 0, 0, flags
    keep = [_f(2048), _f(64), _f(128), _f(64), _f(2048), _f(2048)]
    a.x, a.wq, a.wkv, a.wp, a.y, a.pe = [t.data_ptr() for t in keep]
    a.ln_w = a.ln_b = keep[2].data_ptr()
    if save:
        sv = [_f(2048) for _ in range(5)]
        keep += sv
        a.q, a.k, a.v, a.o, a.lse = [t.data_ptr() for t in sv]
    return a, keep


def _ffn_args(flags, save, x):
    from ecg_denoise_b200 import _lib
    f = _lib.STRUCTS["rl_ffn_fwd_args"]()
    f.B, f.L, f.C, f.le_mode, f.flags = 1, 256, 8, 0, flags
    keep = [_f(256), _f(256), _f(2048), _f(64)]
    f.x, f.w1, f.w2, f.y = x, keep[0].data_ptr(), keep[1].data_ptr(), keep[2].data_ptr()
    f.ln_w = f.ln_b = keep[3].data_ptr()
    if save:
        keep.append(_f(8192))
        f.h = keep[-1].data_ptr()
    return f, keep


def test_abi_rejections():
    from ecg_denoise_b200 import _lib, engine
    from ecg_denoise_b200.ops import _stream
    lib = _lib.load()
    st = ctypes.c_void_p(_stream())
    T, PR = _lib.RL_F_TF32, _lib.RL_F_PRENORM | _lib.RL_F_RESIDUAL

    def rejected(rc):
        assert rc == _lib.RL_ERR_SHAPE
        with pytest.raises(_lib.RalenetError):
            _lib.check(rc)

    # net_fwd with RL_NET_TF32 and save = 1; save = 0 (also with RL_NET_DETERMINISTIC) runs and equals the module
    m = _model("rw", 1, 2023)
    x = torch.randn(5, 2, 256, device="cuda")
    plan = m._plan
    plan.ensure(x.device)
    plan.refresh_requires_grad()
    out = torch.empty(5, 2, 256, device="cuda")

    def net_fwd(save, flags):
        ws = torch.empty(engine.workspace_bytes(5, 256, save, flags), device="cuda", dtype=torch.uint8)
        cfg = plan.cfg(5, 256, False, save, ws, flags)
        rc = lib.ralenet_net_fwd(ctypes.byref(cfg), ctypes.byref(plan.P), ctypes.c_void_p(x.data_ptr()),
                                 ctypes.c_void_p(out.data_ptr()), st)
        torch.cuda.synchronize()
        return rc

    rejected(net_fwd(True, _lib.RL_NET_TF32))
    ref = _run(m, x, "tf32")
    for flags in (_lib.RL_NET_TF32, _lib.RL_NET_TF32 | _lib.RL_NET_DETERMINISTIC):
        assert net_fwd(False, flags) == 0 and torch.equal(out, ref)

    # attn_fwd / ffn_fwd / block_fwd: RL_F_TF32 with saved-tensor pointers; block_fwd: halves with different bits
    a, ka = _attn_args(T, save=True)
    rejected(lib.ralenet_attn_fwd(ctypes.byref(a), st))
    f, kf = _ffn_args(T, True, ka[0].data_ptr())
    rejected(lib.ralenet_ffn_fwd(ctypes.byref(f), st))
    a, ka = _attn_args(PR | T, save=True)
    f, kf = _ffn_args(PR | T, False, a.y)
    rejected(lib.ralenet_block_fwd(ctypes.byref(a), ctypes.byref(f), st))
    a, ka = _attn_args(PR | T, save=False)
    f, kf = _ffn_args(PR, False, a.y)
    rejected(lib.ralenet_block_fwd(ctypes.byref(a), ctypes.byref(f), st))

    # attn_bwd / ffn_bwd with RL_F_TF32
    ab = _lib.STRUCTS["rl_attn_bwd_args"]()
    ab.B, ab.L, ab.C, ab.H, ab.flags = 1, 256, 8, 2, T
    rejected(lib.ralenet_attn_bwd(ctypes.byref(ab), st))
    fb = _lib.STRUCTS["rl_ffn_bwd_args"]()
    fb.B, fb.L, fb.C, fb.flags = 1, 256, 8, T
    rejected(lib.ralenet_ffn_bwd(ctypes.byref(fb), st))
    torch.cuda.synchronize()
