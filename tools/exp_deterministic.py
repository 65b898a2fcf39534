"""Cost of the deterministic mode (FusedTrainer(deterministic=True), RL_NET_DETERMINISTIC) against the default mode.

For each batch size: both graphed trainers on the same model weights and the same device-synthesised batches, timed in
alternating rounds (CUDA events around `--steps` replays, after a warm-up of both), median and spread per mode; the
extra workspace bytes; and the live per-kernel table (un-graphed step, one event pair per launch, on one stream) of both
modes, whose difference names the kernels the deterministic mode adds or slows.  The card name and power limit are
read in the same run.

usage: python tools/exp_deterministic.py [--batches 256 4096] [--rounds 5] [--steps 30] [--out DIR]
(--out DIR also writes the whole report, per-kernel diff included, to DIR/exp_deterministic.json)
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
from ecg_denoise_b200.engine import FusedTrainer, workspace_bytes  # noqa: E402
from ecg_denoise_b200.model import transformer  # noqa: E402
from ecg_denoise_b200.synth_device import DeviceSynth  # noqa: E402
from oracle import synth_weights as SW  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return q


def trainer(det: bool, sd, B: int):
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    tr = FusedTrainer(m, lr=1e-3, use_graph=True, deterministic=det)
    return tr, DeviceSynth(B, 2, 256, seed=2023, kind="emb", snr_db=-4.0)


def timed(tr, sy, steps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        tr.step_synth(sy)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def kernel_table(det: bool, sd, B: int, reps: int = 3):
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    tr = FusedTrainer(m, lr=1e-3, use_graph=False, deterministic=det)
    sy = DeviceSynth(B, 2, 256, seed=2023, kind="emb", snr_db=-4.0)
    tr.step_synth(sy)
    lib = _lib.load()
    agg = {}
    n_max = 8192
    for _ in range(reps):
        torch.cuda.synchronize()
        _lib.check(lib.ralenet_profile_begin(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        tr.step_synth(sy)
        labels = ctypes.create_string_buffer(n_max * 48)
        ms = (ctypes.c_float * n_max)()
        n = lib.ralenet_profile_end(labels, 48, ms, n_max)
        for i in range(n):
            lab = labels.raw[i * 48:(i + 1) * 48].split(b"\0")[0].decode()
            e = agg.setdefault(lab, [0, 0.0])
            e[0] += 1
            e[1] += ms[i]
    return {k: {"launches": v[0] // reps, "ms_per_step": v[1] / reps} for k, v in agg.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 4096])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "exp_deterministic.py needs the B200"
    sd = SW.make_state_dict("rw", 1, 2023)
    report = {"card": card(), "batches": {}}
    print("card:", report["card"])
    for B in args.batches:
        steps = max(3, args.steps * 256 // B)
        trs = {det: trainer(det, sd, B) for det in (False, True)}
        for det, (tr, sy) in trs.items():
            timed(tr, sy, 3)                      # capture + warm-up
        times = {False: [], True: []}
        for r in range(args.rounds):
            order = (False, True) if r % 2 == 0 else (True, False)
            for det in order:
                times[det].append(timed(*trs[det], steps))
        for tr, _ in trs.values():
            tr.close()
        del trs
        torch.cuda.empty_cache()
        extra = workspace_bytes(B, 256, True, _lib.RL_NET_DETERMINISTIC) - workspace_bytes(B, 256, True)
        tabs = {det: kernel_table(det, sd, B) for det in (False, True)}
        rows = []
        for k in sorted(set(tabs[False]) | set(tabs[True])):
            a = tabs[False].get(k, {"launches": 0, "ms_per_step": 0.0})
            b = tabs[True].get(k, {"launches": 0, "ms_per_step": 0.0})
            rows.append((k, a["launches"], b["launches"], a["ms_per_step"], b["ms_per_step"]))
        rows.sort(key=lambda r: -abs(r[4] - r[3]))
        med = {det: statistics.median(v) for det, v in times.items()}
        rec = {"steps_per_round": steps, "ms_default": times[False], "ms_deterministic": times[True],
               "median_default": med[False], "median_deterministic": med[True],
               "spread_default": max(times[False]) - min(times[False]),
               "spread_deterministic": max(times[True]) - min(times[True]),
               "overhead_pct": 100.0 * (med[True] / med[False] - 1.0), "extra_workspace_bytes": extra,
               "kernel_diff": [{"kernel": k, "launches_default": la, "launches_det": lb, "ms_default": ta,
                                "ms_det": tb} for k, la, lb, ta, tb in rows]}
        report["batches"][str(B)] = rec
        print(f"B={B}: default {med[False]:.3f} ms (spread {rec['spread_default']:.3f}), deterministic "
              f"{med[True]:.3f} ms (spread {rec['spread_deterministic']:.3f}) -> {rec['overhead_pct']:+.1f} %, "
              f"extra workspace {extra / 2**20:.1f} MiB")
        print("  per-kernel (live table, eager step): kernel, launches default/det, ms default/det")
        for k, la, lb, ta, tb in rows[:12]:
            print(f"    {k:40s} {la:4d} {lb:4d} {ta:8.3f} {tb:8.3f}")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "exp_deterministic.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
