"""Long-record inference: records -> z-normalised windows -> RA-LENet -> stitched records, all on the GPU.

The reference handles a 30-min record by cutting it into independent 256-sample windows on the host
(local_utils/local_utils.py:47-65, 116-130, np_norm :261-266); windows are independent, so records are sharded
across ranks with no communication (SURVEY.md section 8e).  `denoise_records` does the cut, the per-lead
z-normalisation, the batched eval-mode forward and an overlap-add stitch with hand-written kernels (records.cu).
"""
from __future__ import annotations

import contextlib
import ctypes
from typing import Optional

import torch

from . import _lib
from .engine import check_precision
from .ops import _chk, _stream


def _c(ptr):
    return ctypes.c_void_p(ptr)


def windows_per_record(T: int, window: int = 256, stride: int = 256) -> int:
    return int(_lib.load().ralenet_windows_per_record(ctypes.c_int64(T), window, stride))


def records_to_windows(x: torch.Tensor, window: int = 256, stride: int = 256, znorm: bool = True):
    """x: (R, C, T) CUDA fp32 -> (windows (R*nper, C, window), stats (R*C, 2) or None)."""
    x = _chk(x, "records")
    R, C, T = x.shape
    lib = _lib.load()
    nper = windows_per_record(T, window, stride)
    if nper <= 0:
        raise _lib.RalenetError(f"record length {T} shorter than one window ({window})")
    stats = None
    if znorm:
        stats = torch.empty(R * C, 2, device=x.device, dtype=torch.float32)
        _lib.check(lib.ralenet_record_stats(_c(x.data_ptr()), R * C, ctypes.c_int64(T), _c(stats.data_ptr()),
                                            _c(_stream())))
    win = torch.empty(R * nper, C, window, device=x.device, dtype=torch.float32)
    _lib.check(lib.ralenet_window_gather(_c(x.data_ptr()), _c(stats.data_ptr() if stats is not None else None),
                                         _c(win.data_ptr()), R, C, ctypes.c_int64(T), window, stride, _c(_stream())))
    return win, stats


def windows_to_records(win: torch.Tensor, x: torch.Tensor, stats: Optional[torch.Tensor], stride: int = 256):
    """inverse of records_to_windows: overlap-add average, de-normalise; uncovered tail samples come from x."""
    win, x = _chk(win, "windows"), _chk(x, "records")
    R, C, T = x.shape
    window = win.shape[-1]
    y = torch.empty_like(x)
    _lib.check(_lib.load().ralenet_window_scatter(
        _c(win.data_ptr()), _c(x.data_ptr()), _c(stats.data_ptr() if stats is not None else None), _c(y.data_ptr()),
        R, C, ctypes.c_int64(T), window, stride, _c(_stream())))
    return y


@contextlib.contextmanager
def precision_scope(model, precision: Optional[str]):
    """for the body: with precision "fp32" or "tf32", that inference_precision on every RA-LENet module inside `model`
    (e.g. the core of a 12-lead `newrale`), restored afterwards; None changes nothing."""
    from .model._blocks import _RalenetBase
    cores = []
    if precision is not None:
        check_precision(precision)
        cores = [(m, m.inference_precision) for m in model.modules() if isinstance(m, _RalenetBase)]
    try:
        for m, _ in cores:
            m.inference_precision = precision
        yield
    finally:
        for m, p in cores:
            m.inference_precision = p


@torch.no_grad()
def denoise_records(model, records: torch.Tensor, window: int = 256, stride: int = 256, batch: int = 8192,
                    znorm: bool = True, stitch: bool = True, precision: Optional[str] = None):
    """Denoise (R, 2, T) records with an RA-LENet `model` in eval mode.  Returns the stitched records
    (R, 2, T), or the denoised windows (R*nper, 2, window) when stitch=False.  Data-parallel use: give each rank
    its own slice of the records -- no communication is needed.
    precision: None keeps the inference_precision of every RA-LENet module inside `model`; "fp32" or "tf32" sets it
    on all of them (e.g. the core of a 12-lead `newrale`) for this call and restores it afterwards."""
    was_training = model.training
    with precision_scope(model, precision):
        model.eval()
        try:
            win, stats = records_to_windows(records, window, stride, znorm)
            out = torch.empty_like(win)
            for i in range(0, win.shape[0], batch):
                out[i:i + batch] = model(win[i:i + batch])
            return windows_to_records(out, records, stats, stride) if stitch else out
        finally:
            model.train(was_training)
