"""Cost of the deterministic 12-lead fine-tune (FineTuneTrainer(deterministic=True)) against the default mode.

For each batch size: both graphed trainers on the same newrale weights and the same device-synthesised 12-lead batches,
timed in alternating rounds (CUDA events around `--steps` replays, after a warm-up of both), median and spread per
mode, and the extra bytes the deterministic mode allocates: the core's RL_NET_DETERMINISTIC workspace (sized for every
core parameter although the fine-tune freezes them all), the four convolution slabs and the loss partials.  The card
name, power limit and max SM clock are read in the same run.

usage: python tools/exp_deterministic_finetune.py [--batches 1280 256] [--rounds 7] [--steps 20] [--out DIR]
(--out DIR also writes the report to DIR/exp_deterministic_finetune.json)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from ecg_denoise_b200 import _lib  # noqa: E402
from ecg_denoise_b200.engine import FineTuneTrainer, workspace_bytes  # noqa: E402
from ecg_denoise_b200.model import ralenet_12leads as TW  # noqa: E402
from ecg_denoise_b200.synth_device import DeviceSynth  # noqa: E402
from oracle import synth_weights as SW  # noqa: E402

LAYERS = [(12, 6, 13), (6, 2, 13), (2, 6, 13), (6, 12, 13)]      # newrale's convolutions (Cin, Cout, K)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return q


def extra_bytes(B: int, L: int = 256) -> dict:
    lib = _lib.load()
    core = workspace_bytes(B, L, True, _lib.RL_NET_DETERMINISTIC) - workspace_bytes(B, L, True)
    slabs = sum(int(lib.ralenet_conv1d_slab_bytes(B, *s)) for s in LAYERS)
    return {"core_workspace": core, "conv_slabs": slabs, "loss_partials": 4 * B, "total": core + slabs + 4 * B}


def trainer(det: bool, sd, B: int):
    m = TW.newrale(TW.ralenet(high_level_enhence=True))
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    tr = FineTuneTrainer(m, lr=1e-3, use_graph=True, deterministic=det)
    return tr, DeviceSynth(B, 12, 256, seed=2023, kind="emb", snr_db=-4.0)


def timed(tr, sy, steps: int) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        tr.step_synth(sy)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[1280, 256])
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "exp_deterministic_finetune.py needs the B200"
    sd = SW.make_newrale_state_dict(2023)
    report = {"card": card(), "batches": {}}
    print("card:", report["card"])
    for B in args.batches:
        steps = max(5, args.steps * 1280 // B)
        trs = {det: trainer(det, sd, B) for det in (False, True)}
        for tr, sy in trs.values():
            timed(tr, sy, 3)                      # capture + warm-up
        times = {False: [], True: []}
        for r in range(args.rounds):
            for det in ((False, True) if r % 2 == 0 else (True, False)):
                times[det].append(timed(*trs[det], steps))
        for tr, _ in trs.values():
            tr.close()
        del trs
        torch.cuda.empty_cache()
        med = {det: statistics.median(v) for det, v in times.items()}
        extra = extra_bytes(B)
        rec = {"steps_per_round": steps, "ms_default": times[False], "ms_deterministic": times[True],
               "median_default": med[False], "median_deterministic": med[True],
               "spread_default": max(times[False]) - min(times[False]),
               "spread_deterministic": max(times[True]) - min(times[True]),
               "overhead_pct": 100.0 * (med[True] / med[False] - 1.0), "extra_bytes": extra}
        report["batches"][str(B)] = rec
        print(f"B={B} x 12 x 256: default {med[False]:.3f} ms (spread {rec['spread_default']:.3f}), deterministic "
              f"{med[True]:.3f} ms (spread {rec['spread_deterministic']:.3f}) -> {rec['overhead_pct']:+.1f} %; extra "
              f"bytes: core workspace {extra['core_workspace'] / 2**20:.1f} MiB, conv slabs "
              f"{extra['conv_slabs'] / 2**20:.2f} MiB, loss partials {extra['loss_partials']} B")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "exp_deterministic_finetune.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
