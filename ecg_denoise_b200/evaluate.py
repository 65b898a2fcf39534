"""Held-out evaluation on the device (csrc/records.cu record_enumerate_kernel, csrc/stem_head.cu eval_*_kernel): every
window of a clean test bank at every SNR level, exactly once, with a fixed noise pairing, reduced to per-level SNR and
RMSE figures on the GPU -- the per-epoch test loop of the reference without a host loop.

The reference evaluates after every epoch (denoise_train.py:66-81): model.eval() over the test loader, the per-window
SNR and RMSE of local_utils/evaluate.py:27-29, 49-51, and one SNR / RMSE line per noise type and intensity
(denoise_train.py:100-101; one test set per intensity, dict_data/{m4,m2,0,p2,p4}).  `RecordEvaluator.run(model)` does
the same from two banks that stay in HBM:

  * record_enumerate_kernel takes item e = g * n_snr + lvl of the (grid window, level) set for every slot, in order
    (slot i of batch k on rank r: e = k * world * B + r * B + i); the noise window of a pair is hashed from
    (seed, g, lvl) alone, so every run, epoch and rank split sees the same noisy test set;
  * ralenet_snr_mix adds the noise at the level; the model runs its no-grad eval forward;
  * ralenet_eval_metrics adds (count, snr_in, snr_out, rmse) per level into an fp64 accumulator in a fixed order and
    bumps the batch counter, so with use_graph=True one captured step is replayed `steps` times.

The last batch may run past the end of the set: its extra slots are zero windows marked level -1 and add nothing.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Dict, Optional, Sequence, Union

import torch

from . import _lib
from .inference import precision_scope
from .ops import _stream
from .record_sampler import _RecordBanks


@dataclasses.dataclass
class EvalResult:
    """Per-level means over the evaluated windows, keyed by the level in dB: input SNR, output SNR, their difference
    (SNR improvement) and RMSE (local_utils/evaluate.py), the window count per level, and `acc`, the (n_snr, 4)
    float64 device accumulator (count, sum snr_in, sum snr_out, sum rmse) they come from."""
    snr_in: Dict[float, float]
    snr_out: Dict[float, float]
    snr_imp: Dict[float, float]
    rmse: Dict[float, float]
    count: Dict[float, int]
    acc: torch.Tensor


class RecordEvaluator(_RecordBanks):
    """Every grid window of a held-out clean bank at every SNR level, once, evaluated on the device.

    records: (R, leads, T) CUDA fp32 contiguous; noise: (N, 1 or leads, Tn) on the same device; batch: windows per step
    on this rank; window, stride (None = window), znorm, rank / world: as in record_sampler.RecordSampler.  snr_db: the
    levels in dB (distinct), each applied to every window.  seed keys the noise pairing.
    `steps` = ceil(R * nper * n_snr / (world * batch)) steps cover the set; fill(k) draws step k into `noisy` / `clean`
    (`meta`, `snr`, `level` describe it; `valid` = level >= 0).
    """
    _WHO = "RecordEvaluator"

    def __init__(self, records: torch.Tensor, noise: torch.Tensor, batch: int, window: int = 256,
                 stride: Optional[int] = None, snr_db: Union[float, Sequence[float]] = (-4, -2, 0, 2, 4),
                 znorm: bool = True, seed: int = 2023, rank: Optional[int] = None, world: Optional[int] = None):
        super().__init__("rl_enum_args", records, noise, batch, window, stride, snr_db, znorm, seed, rank, world)
        dev, B = self.device, self.B
        self.clean = torch.empty(B, self.leads, self.L, device=dev, dtype=torch.float32)
        self.noisy = torch.empty_like(self.clean)
        self.level = torch.empty(B, device=dev, dtype=torch.int32)
        self.counter = torch.zeros(1, device=dev, dtype=torch.int32)
        self.acc = torch.zeros(len(self.levels), 4, device=dev, dtype=torch.float64)
        self._partials = torch.empty(B, 4, device=dev, dtype=torch.float64)
        # per-window values of the most recent step (0 in slots past the end of the set)
        self.window_snr_in = torch.empty(B, device=dev, dtype=torch.float32)
        self.window_snr_out = torch.empty(B, device=dev, dtype=torch.float32)
        self.window_rmse = torch.empty(B, device=dev, dtype=torch.float32)
        a = self._args
        a.clean_out, a.level, a.counter = self.clean.data_ptr(), self.level.data_ptr(), self.counter.data_ptr()
        m = _lib.STRUCTS["rl_eval_args"]()
        m.clean, m.noisy, m.level = self.clean.data_ptr(), self.noisy.data_ptr(), self.level.data_ptr()
        m.snr_in, m.snr_out, m.rmse = (self.window_snr_in.data_ptr(), self.window_snr_out.data_ptr(),
                                       self.window_rmse.data_ptr())
        m.partials, m.acc, m.counter = self._partials.data_ptr(), self.acc.data_ptr(), self.counter.data_ptr()
        m.B, m.per, m.n_snr = B, self.leads * self.L, len(self.levels)
        self._margs = m

    def _check_grid(self, R, nper, levels, batch, world):
        if len(set(levels)) != len(levels):
            raise ValueError(f"RecordEvaluator: snr_db {levels} repeats a level (the results are keyed by level)")
        self.levels = tuple(levels)
        self.n_items = R * nper * len(levels)
        self.steps = math.ceil(self.n_items / (world * batch))

    @property
    def valid(self) -> torch.Tensor:
        return self.level >= 0

    # -- the three pieces of one step --------------------------------------------------------------------------------
    def _draw(self):
        st = _stream()
        _lib.call("ralenet_record_enumerate", self._args, st)
        _lib.check(_lib.load().ralenet_snr_mix(self.clean.data_ptr(), self.noise.data_ptr(), self.snr.data_ptr(),
                                               self.noisy.data_ptr(), self.B, self.leads * self.L, st))

    def _step(self, model):
        self._draw()
        pred = model(self.noisy)
        if tuple(pred.shape) != tuple(self.noisy.shape) or pred.dtype != torch.float32 or not pred.is_contiguous():
            raise _lib.RalenetError(f"RecordEvaluator: the model returned {pred.dtype} {tuple(pred.shape)}, expected "
                                    f"contiguous float32 {tuple(self.noisy.shape)}")
        self._margs.pred = pred.data_ptr()
        _lib.call("ralenet_eval_metrics", self._margs, _stream())

    def fill(self, counter: int = 0):
        """draw step `counter` into `clean` / `noisy` (and `meta`, `snr`, `level`) without evaluating it."""
        self.counter.fill_(int(counter))
        self._draw()

    # -- evaluation ------------------------------------------------------------------------------------------------
    def _check_model(self, model):
        from .model._blocks import _RalenetBase
        from .model.ralenet_12leads import newrale
        if isinstance(model, _RalenetBase):
            cin = model.conv1[0].in_channels
        elif isinstance(model, newrale):
            cin = model.conv1.in_channels
        else:
            raise TypeError(f"RecordEvaluator: {type(model).__name__} is not an RA-LENet model (the three ralenet "
                            "classes or newrale)")
        if cin != self.leads:
            raise ValueError(f"RecordEvaluator: the banks have {self.leads} leads, the model takes {cin}")

    def run(self, model, precision: Optional[str] = None, use_graph: bool = True) -> EvalResult:
        """Evaluate `model` on the whole set: eval mode and the no-grad forward, no autograd node; parameters and
        BatchNorm buffers are not touched, and every module's training flag is restored afterwards.  precision: None
        keeps each RA-LENet module's inference_precision, "fp32" / "tf32" applies to this call (as denoise_records).
        use_graph: capture one step (draw, mix, forward, metrics) and replay it `steps` times; False runs the same
        calls eagerly, with a bit-identical result.  Under torch.distributed with world > 1 the accumulator is summed
        over the ranks with one all_reduce (fp64; the symmetric-memory exchange of comm.py carries fp32).  The host
        reads the result once, at the end."""
        self._check_model(model)
        modes = [(m, m.training) for m in model.modules()]
        with precision_scope(model, precision), torch.no_grad():
            model.eval()
            try:
                if use_graph:
                    graph = self._capture(model)
                    self.acc.zero_()
                    self.counter.zero_()
                    for _ in range(self.steps):
                        graph.replay()
                else:
                    self.acc.zero_()
                    self.counter.zero_()
                    for _ in range(self.steps):
                        self._step(model)
            finally:
                for m, t in modes:
                    m.training = t
        dist = torch.distributed
        if self.world > 1 and dist.is_available() and dist.is_initialized() and dist.get_world_size() == self.world:
            dist.all_reduce(self.acc)
        host = self.acc.cpu().tolist()
        res = EvalResult({}, {}, {}, {}, {}, self.acc)
        for lv, (n, s_in, s_out, s_rmse) in zip(self.levels, host):
            res.count[lv] = int(n)
            res.snr_in[lv] = s_in / n if n else math.nan
            res.snr_out[lv] = s_out / n if n else math.nan
            res.snr_imp[lv] = res.snr_out[lv] - res.snr_in[lv]
            res.rmse[lv] = s_rmse / n if n else math.nan
        return res

    def _capture(self, model) -> torch.cuda.CUDAGraph:
        # the warm-up step does the first-call set-up (flat parameters, positional tables, kernel attributes) outside
        # the capture; run() zeroes what it accumulated
        s = torch.cuda.Stream(self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            self.counter.zero_()
            self._step(model)
        torch.cuda.current_stream(self.device).wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            self._step(model)
        return graph
