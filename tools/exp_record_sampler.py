"""Cost of the device-resident record sampler (record_sampler.RecordSampler) inside the graphed training step.

For each batch size, three graphed FusedTrainer steps on the same model weights, timed in alternating rounds (CUDA
events around `--steps` replays, after a warm-up of each):
  static  -- step(x, t) on a fixed device batch (two device-to-device copies into the static buffers per step);
  synth   -- step_synth(DeviceSynth): synthetic windows drawn inside the graph;
  records -- step_synth(RecordSampler): windows of a record bank of 48 x 2 x 650,000 samples (MIT-BIH-shaped,
             250 MB, larger than the 126 MB L2) paired with windows of a noise bank of 3 x 2 x 650,000 samples at
             SNR levels -4..4 dB, drawn inside the graph.
Then the kernel times of the sampler alone (ralenet_profile_*: one event pair per launch, `--fills` fills of the
batch): record_sample_kernel and snr_mix_kernel, and their sum as a share of the median record-fed step.
The card name and power limit are read in the same run.

usage: python tools/exp_record_sampler.py [--batches 256 4096] [--rounds 3] [--steps 30] [--out DIR]
(--out DIR also writes the report to DIR/exp_record_sampler.json)
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from ecg_denoise_b200 import _lib  # noqa: E402
from ecg_denoise_b200.engine import FusedTrainer  # noqa: E402
from ecg_denoise_b200.model import transformer  # noqa: E402
from ecg_denoise_b200.record_sampler import RecordSampler  # noqa: E402
from ecg_denoise_b200.synth_device import DeviceSynth  # noqa: E402
from oracle import synth_weights as SW  # noqa: E402

FORMS = ("static", "synth", "records")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return q


def trainer(sd):
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(sd, strict=True)
    return FusedTrainer(m.cuda().train(), lr=1e-3, use_graph=True)


def timed(step, steps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def sampler_kernels(sp, fills: int):
    """ms per fill of each kernel the sampler launches (record_sample_kernel, snr_mix_kernel)"""
    lib = _lib.load()
    noisy, clean = sp.batch(0)
    ctr = torch.zeros(1, device="cuda", dtype=torch.int32)
    torch.cuda.synchronize()
    n_max, stride = 4 * fills, 48
    labels, ms = ctypes.create_string_buffer(n_max * stride), (ctypes.c_float * n_max)()
    _lib.check(lib.ralenet_profile_begin(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    for _ in range(fills):
        sp.fill(noisy, clean, ctr)
        ctr += 1                           # a new batch per fill, as in training
    got = lib.ralenet_profile_end(labels, stride, ms, n_max)
    _lib.check(0 if got > 0 else -3)
    agg = {}
    for i in range(got):
        lab = labels.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode()
        agg[lab] = agg.get(lab, 0.0) + float(ms[i]) / fills
    return agg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 4096])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--fills", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "exp_record_sampler.py needs the B200"
    report = {"card": card(), "record_bank": [48, 2, 650000], "noise_bank": [3, 2, 650000], "batches": {}}
    print("card:", report["card"])
    g = torch.Generator(device="cuda").manual_seed(2023)
    recs = torch.randn(48, 2, 650000, device="cuda", generator=g) * 0.3 + 0.1
    noise = torch.randn(3, 2, 650000, device="cuda", generator=g)
    sd = SW.make_state_dict("rw", 1, 2023)
    for B in args.batches:
        steps = max(10, args.steps * 256 // B)
        sp = RecordSampler(recs, noise, B, seed=2023)
        sy = DeviceSynth(B, 2, 256, seed=2023, kind="emb", snr_db=-4.0)
        x, t = sy.batch()
        trs = {f: trainer(sd) for f in FORMS}
        run = {"static": lambda: trs["static"].step(x, t), "synth": lambda: trs["synth"].step_synth(sy),
               "records": lambda: trs["records"].step_synth(sp)}
        for f in FORMS:
            timed(run[f], 3)                   # capture + warm-up
        times = {f: [] for f in FORMS}
        for r in range(args.rounds):
            for f in (FORMS if r % 2 == 0 else FORMS[::-1]):
                times[f].append(timed(run[f], steps))
        for tr in trs.values():
            tr.close()
        del trs
        torch.cuda.empty_cache()
        med = {f: statistics.median(v) for f, v in times.items()}
        kern = sampler_kernels(sp, args.fills)
        k_ms = kern.get("record_sample_kernel", 0.0) + kern.get("snr_mix_kernel", 0.0)
        rec = {"steps_per_round": steps, "steps_per_epoch": sp.steps_per_epoch,
               "ms": times, "median_ms": med, "spread_ms": {f: max(v) - min(v) for f, v in times.items()},
               "sampler_kernel_ms": kern, "sampler_ms": k_ms, "sampler_pct_of_step": 100.0 * k_ms / med["records"]}
        report["batches"][str(B)] = rec
        print(f"B={B} ({steps} steps per round, {args.rounds} rounds):")
        for f in FORMS:
            print(f"  {f:8s} median {med[f]:8.3f} ms  (spread {rec['spread_ms'][f]:.3f})  "
                  f"{100.0 * (med[f] / med['static'] - 1.0):+6.2f} % vs static")
        for lab, v in sorted(kern.items()):
            print(f"  kernel {lab:28s} {1e3 * v:8.2f} us per fill")
        print(f"  sampler + mix: {1e3 * k_ms:.2f} us = {rec['sampler_pct_of_step']:.3f} % of the record-fed step")
    report["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "exp_record_sampler.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
