"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

from contextlib import contextmanager

import numpy as np
import torch

SUB = 32
STRIDE_PRIME = 37

CASES = {
    # tag: (variant, le, seed, x key, target key)
    "rw_le": ("rw", 1, 2023, "x", "target"),
    "rw_mlp": ("rw", 0, 2024, "x", "target"),
    "nra": ("nra", 1, 2025, "x", "target"),
    "nra512": ("nra", 1, 2025, "x512", "target512"),
}


def subsample(t: torch.Tensor) -> np.ndarray:
    """must mirror oracle/make_golden.py::subsample."""
    f = t.detach().reshape(-1).to(torch.float64).cpu().numpy()
    if f.size <= SUB:
        return f.copy()
    idx = (np.arange(SUB) * STRIDE_PRIME * (f.size // SUB // STRIDE_PRIME + 1)) % f.size
    return f[idx].copy()


def pack(t: torch.Tensor) -> np.ndarray:
    t = t.detach().to(torch.float64).cpu()
    return np.concatenate([[t.sum().item(), t.norm().item()], subsample(t)])


def unpack_golden(names, packed, shapes):
    """split the packed per-parameter golden vector -> {name: (sum, norm, samples)}."""
    out, o = {}, 0
    for n in names:
        k = min(int(np.prod(shapes[n])) if len(shapes[n]) else 1, SUB)
        out[n] = (packed[o], packed[o + 1], packed[o + 2:o + 2 + k])
        o += 2 + k
    assert o == len(packed)
    return out


def rel_rms_err(a, b) -> float:
    """max |a-b| / (|b| + rms(b)) -- the tolerance definition of BASELINE.md section 3."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    rms = np.sqrt((b * b).mean()) + 1e-300
    return float(np.max(np.abs(a - b) / (np.abs(b) + rms)))


def check_packed(got: torch.Tensor, gold, rtol: float, name: str):
    gsum, gnorm, gsamp = gold
    p = pack(got)
    scale = gnorm + 1e-30
    assert abs(p[1] - gnorm) <= rtol * scale, f"{name}: norm {p[1]} vs {gnorm}"
    n_el = got.numel()
    assert abs(p[0] - gsum) <= rtol * scale * np.sqrt(n_el), f"{name}: sum {p[0]} vs {gsum}"
    rms = gnorm / np.sqrt(n_el)
    err = np.max(np.abs(p[2:] - gsamp) / (np.abs(gsamp) + rms + 1e-30))
    assert err <= rtol, f"{name}: sample rel err {err:.3e} > {rtol}"


@contextmanager
def switches(mode):
    """kernel-selection switches: 'default', 'reg2' (register-tile GEMMs for every group), 'mma' (mma.sync GEMMs)."""
    from ecg_denoise_b200 import _lib
    lib = _lib.load()
    prev_reg, prev_umma = lib.ralenet_set_wgrad_reg(1), lib.ralenet_set_wgrad_umma(1)
    if mode == "reg2":
        lib.ralenet_set_wgrad_reg(2)
    elif mode == "mma":
        lib.ralenet_set_wgrad_reg(0)
        lib.ralenet_set_wgrad_umma(0)
    try:
        yield
    finally:
        lib.ralenet_set_wgrad_reg(prev_reg)
        lib.ralenet_set_wgrad_umma(prev_umma)
