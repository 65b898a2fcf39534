"""Device-resident record sampler (csrc/records.cu + the SNR-mix kernel): training batches cut from REAL records on
the GPU, inside the training step's CUDA graph -- the real-data half of SURVEY.md section 8 f3.

The reference prepares its pairs on the host: MIT-BIH records z-normalised per lead (np_norm,
local_utils/local_utils.py:261-266), cut into windows with range(0, T, stride) (:47-65), NSTDB noise records mixed in
at a target SNR (single_snr_noise_add, :176-192), then shuffled by a DataLoader (main.py:45-60).  `RecordSampler.fill`
does all of it on the device from two record banks that stay resident in HBM:

  * record_sample_kernel picks, for every slot of the batch, a window of the clean bank (z-normalised with
    statistics computed once, exactly like records_to_windows), a window of the noise bank and an SNR level;
  * ralenet_snr_mix (the pinned reference formula) adds the noise at that level.

Every draw is a pure function of (seed, counter, global slot).  An epoch is one pass over the grid of R * nper
windows in a keyed order that changes with the epoch (drop-last); stride = window is the reference's cut, stride = 1
random crops without replacement.  The counter is the batch index: `FusedTrainer.step_synth(sampler)` and
`FineTuneTrainer.step_synth(sampler)` pass the Adam step counter, so every graph replay trains on the next batch.
Data-parallel ranks draw disjoint slices of the same world batch: the slices of `world` ranks of B windows each,
put together, are the batch of world * B windows a single process would draw.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Union

import torch

from . import _lib
from .inference import windows_per_record
from .ops import _stream


def steps_per_epoch(R: int, T: int, window: int, stride: int, batch: int, world: int = 1) -> int:
    """floor(R * nper / (world * batch)): the full batches of one pass over the grid (the remainder is dropped)."""
    return R * windows_per_record(T, window, stride) // (world * batch)


def _bank(t, name: str, who: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or t.dim() != 3:
        raise ValueError(f"{who}: {name} must be a 3-D tensor (records, leads, samples), "
                         f"got {getattr(t, 'shape', type(t).__name__)}")
    return t


class _RecordBanks:
    """What the device batch sources over a clean and a noise record bank share: argument checks (ValueError for
    shapes and values, before any device work; RalenetError for placement), the per-(record, lead) z-normalisation
    statistics, the level table, the per-slot noise / level / meta buffers and the C argument struct, whose bank fields
    rl_sample_args and rl_enum_args have in common.  Subclasses name themselves in _WHO (for messages) and check the
    size of the grid in _check_grid."""
    _WHO: str

    def __init__(self, struct: str, records, noise, batch, window, stride, snr_db, znorm, seed, rank, world):
        who = self._WHO
        records, noise = _bank(records, "records", who), _bank(noise, "noise", who)
        R, leads, T = records.shape
        N, noise_leads, Tn = noise.shape
        stride = window if stride is None else stride
        levels = [float(snr_db)] if isinstance(snr_db, (int, float)) else [float(s) for s in snr_db]
        if world is None or rank is None:
            dist = torch.distributed.is_available() and torch.distributed.is_initialized()
            world = (torch.distributed.get_world_size() if dist else 1) if world is None else world
            rank = (torch.distributed.get_rank() if dist else 0) if rank is None else rank
        batch, window, stride, world, rank = int(batch), int(window), int(stride), int(world), int(rank)
        if not 1 <= leads <= 12:
            raise ValueError(f"{who}: records have {leads} leads; 1 to 12 are supported")
        if noise_leads not in (1, leads):
            raise ValueError(f"{who}: noise has {noise_leads} leads; it needs 1 or {leads} (as the records)")
        if batch < 1 or window < 1 or stride < 1:
            raise ValueError(f"{who}: batch={batch}, window={window}, stride={stride} must be positive")
        if window > T or window > Tn:
            raise ValueError(f"{who}: window {window} is longer than the records ({T}) or the noise ({Tn})")
        if not levels:
            raise ValueError(f"{who}: snr_db needs at least one level")
        if not 0 <= rank < world:
            raise ValueError(f"{who}: rank {rank} is not in [0, world={world})")
        self._check_grid(R, windows_per_record(T, window, stride), levels, batch, world)
        for t, name in ((records, "records"), (noise, "noise")):
            if not t.is_cuda:
                raise _lib.RalenetError(f"{who}: {name} is on {t.device}; the banks are read on a CUDA B200 device "
                                        "(no CPU fallback)")
            if t.dtype != torch.float32:
                raise _lib.RalenetError(f"{who}: {name} has dtype {t.dtype}; the kernel reads float32")
            if not t.is_contiguous():
                raise _lib.RalenetError(f"{who}: {name} must be contiguous (it is read in place)")
        if noise.device != records.device:
            raise _lib.RalenetError(f"{who}: noise is on {noise.device}, records on {records.device}")
        self.device = records.device
        _lib.check_device(self.device.index if self.device.index is not None else torch.cuda.current_device())

        self.records, self.noise_bank = records, noise
        self.B, self.leads, self.L, self.stride, self.seed = batch, leads, window, stride, int(seed)
        self.rank, self.world = rank, world
        self.snr_levels = torch.tensor(levels, device=self.device, dtype=torch.float32)
        lib = _lib.load()
        self.stats = None
        if znorm:
            self.stats = torch.empty(R * leads, 2, device=self.device, dtype=torch.float32)
            _lib.check(lib.ralenet_record_stats(ctypes.c_void_p(records.data_ptr()), R * leads, ctypes.c_int64(T),
                                                ctypes.c_void_p(self.stats.data_ptr()), ctypes.c_void_p(_stream())))
        self.noise = torch.empty(batch, leads, window, device=self.device, dtype=torch.float32)
        self.snr = torch.empty(batch, device=self.device, dtype=torch.float32)
        self.meta = torch.empty(batch, 4, device=self.device, dtype=torch.int32)
        a = _lib.STRUCTS[struct]()
        a.records, a.noise, a.snr_levels = records.data_ptr(), noise.data_ptr(), self.snr_levels.data_ptr()
        a.stats = self.stats.data_ptr() if self.stats is not None else None
        a.noise_out, a.snr_out, a.meta = self.noise.data_ptr(), self.snr.data_ptr(), self.meta.data_ptr()
        a.T, a.Tn, a.seed = T, Tn, self.seed & 0xFFFFFFFFFFFFFFFF
        a.R, a.leads, a.N, a.noise_leads, a.n_snr = R, leads, N, noise_leads, len(levels)
        a.W, a.stride, a.B, a.rank, a.world = window, stride, batch, rank, world
        self._args = a

    def _check_grid(self, R: int, nper: int, levels: list, batch: int, world: int) -> None:
        raise NotImplementedError


class RecordSampler(_RecordBanks):
    """Training windows drawn on the device from a bank of clean records and a bank of noise records.

    records: (R, leads, T) CUDA fp32 contiguous, leads <= 12; noise: (N, noise_leads, Tn) on the same device,
    noise_leads = 1 or leads (clean lead l is paired with noise lead l % noise_leads).
    batch: windows per call on this rank; window: samples per window (the trainer's L); stride: grid step of the
    record cut (None = window); snr_db: one level or a sequence of levels, drawn uniformly per window; znorm: per
    (record, lead) z-normalisation with population statistics (np_norm); rank / world: this process's slice of the
    world batch (default: torch.distributed when it is initialised, else 0 / 1).

    fill(noisy, clean, counter) enqueues the batch of `counter` into two (batch, leads, window) buffers; after it,
    `meta` (batch, 4) int32 holds (record, offset, noise record, noise offset) per window and `snr` (batch,) the
    drawn levels in dB.
    """
    _WHO = "RecordSampler"

    def __init__(self, records: torch.Tensor, noise: torch.Tensor, batch: int, window: int = 256,
                 stride: Optional[int] = None, snr_db: Union[float, Sequence[float]] = (-4, -2, 0, 2, 4),
                 znorm: bool = True, seed: int = 2023, rank: Optional[int] = None, world: Optional[int] = None):
        super().__init__("rl_sample_args", records, noise, batch, window, stride, snr_db, znorm, seed, rank, world)

    def _check_grid(self, R, nper, levels, batch, world):
        spe = R * nper // (world * batch)
        if spe == 0:
            raise ValueError(f"RecordSampler: the grid has {R * nper} windows, fewer than one world batch of "
                             f"{world} x {batch}")
        self.steps_per_epoch = spe

    def _counter(self, counter) -> Optional[torch.Tensor]:
        if counter is None or isinstance(counter, torch.Tensor):
            if counter is not None and (counter.device != self.device or counter.dtype != torch.int32
                                        or counter.numel() < 1):
                raise _lib.RalenetError(f"RecordSampler: counter must be an int32 tensor on {self.device}, got "
                                        f"{counter.dtype} on {counter.device}")
            return counter
        return torch.full((1,), int(counter), device=self.device, dtype=torch.int32)

    def fill(self, noisy: torch.Tensor, clean: torch.Tensor, counter: Union[None, int, torch.Tensor] = None):
        """enqueue the batch of `counter` (device int32 tensor, a Python int, or None = 0) into `noisy`, `clean`:
        (B, leads, window) CUDA fp32 contiguous tensors on the sampler's device.  No host synchronisation, so it can
        be captured in a CUDA graph (with a device counter)."""
        shape = (self.B, self.leads, self.L)
        for t, name in ((noisy, "noisy"), (clean, "clean")):
            if tuple(t.shape) != shape:
                raise ValueError(f"RecordSampler.fill: {name} has shape {tuple(t.shape)}, expected {shape}")
            if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous():
                raise _lib.RalenetError(f"RecordSampler.fill: {name} must be a contiguous float32 tensor on "
                                        f"{self.device}, got {t.dtype} on {t.device}")
        ctr = self._counter(counter)
        a = self._args
        a.clean_out = clean.data_ptr()
        a.counter = ctr.data_ptr() if ctr is not None else None
        lib = _lib.load()
        st = ctypes.c_void_p(_stream())
        _lib.check(lib.ralenet_record_sample(ctypes.byref(a), st))
        _lib.check(lib.ralenet_snr_mix(clean.data_ptr(), self.noise.data_ptr(), self.snr.data_ptr(), noisy.data_ptr(),
                                       self.B, self.leads * self.L, st))

    def batch(self, counter: Union[None, int, torch.Tensor] = None):
        """(noisy, clean) of batch `counter` in new tensors; `meta` and `snr` describe it until the next fill."""
        noisy = torch.empty(self.B, self.leads, self.L, device=self.device, dtype=torch.float32)
        clean = torch.empty_like(noisy)
        self.fill(noisy, clean, counter)
        return noisy, clean
