"""Throughput of the device-resident held-out evaluation (evaluate.RecordEvaluator.run) next to record inference.

Workload: a clean bank of 48 x 2 x 650,000 samples (MIT-BIH-shaped, 250 MB, larger than the 126 MB L2) and a noise
bank of 3 x 2 x 650,000 samples; every one of the 121,872 grid windows at five SNR levels (-4..4 dB), i.e. 609,360
evaluated windows per run, `--batch` windows per step.  Timed with CUDA events around whole `run` calls (graph capture
included), in fp32 and tf32 precision, graph on and off, in alternating rounds after one warm-up run of each; next to it
`denoise_records` on the same clean bank (121,872 windows, same batch) in the same precision.  Reports windows/s per
round, median and spread, checks that graph and eager runs give bit-identical accumulators, and prints the per-level
figures.  The card name and power limit are read in the same run.

usage: python tools/exp_record_eval.py [--batch 4096] [--rounds 3] [--out DIR]
(--out DIR also writes the report to DIR/exp_record_eval.json)
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

from ecg_denoise_b200.evaluate import RecordEvaluator  # noqa: E402
from ecg_denoise_b200.inference import denoise_records  # noqa: E402
from ecg_denoise_b200.model import transformer  # noqa: E402
from oracle import synth_weights as SW  # noqa: E402

LEVELS = (-4.0, -2.0, 0.0, 2.0, 4.0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return q


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "exp_record_eval.py needs the B200"
    report = {"card": card(), "record_bank": [48, 2, 650000], "noise_bank": [3, 2, 650000], "levels": LEVELS,
              "batch": args.batch}
    print("card:", report["card"])
    g = torch.Generator(device="cuda").manual_seed(2023)
    recs = torch.randn(48, 2, 650000, device="cuda", generator=g) * 0.3 + 0.1
    noise = torch.randn(3, 2, 650000, device="cuda", generator=g)
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(SW.make_state_dict("rw", 1, 2023), strict=True)
    model = m.cuda()
    ev = RecordEvaluator(recs, noise, args.batch, snr_db=LEVELS, seed=2023)
    n_eval, n_inf = ev.n_items, 48 * ((650000 - 256) // 256 + 1)
    report.update(eval_windows=n_eval, eval_steps=ev.steps, infer_windows=n_inf)
    forms = {}
    for prec in ("fp32", "tf32"):
        for graph in (True, False):
            forms[f"eval_{prec}_{'graph' if graph else 'eager'}"] = (
                n_eval, lambda p=prec, gr=graph: ev.run(model, precision=p, use_graph=gr))
        forms[f"infer_{prec}"] = (n_inf, lambda p=prec: denoise_records(model, recs, batch=args.batch, precision=p))
    accs = {}
    for name, (_, fn) in forms.items():                      # warm-up: module load, first-call set-up, allocator pool
        _, out = timed(fn)
        if name.startswith("eval"):
            accs[name] = out.acc.clone()
            if name.endswith("graph") and "fp32" in name:
                report["fp32_per_level"] = {str(lv): {"count": out.count[lv], "snr_in": out.snr_in[lv],
                                                      "snr_out": out.snr_out[lv], "snr_imp": out.snr_imp[lv],
                                                      "rmse": out.rmse[lv]} for lv in ev.levels}
        del out
    report["graph_equals_eager"] = {p: bool(torch.equal(accs[f"eval_{p}_graph"], accs[f"eval_{p}_eager"]))
                                    for p in ("fp32", "tf32")}
    rates = {name: [] for name in forms}
    names = list(forms)
    for r in range(args.rounds):
        for name in (names if r % 2 == 0 else names[::-1]):
            n, fn = forms[name]
            sec, _ = timed(fn)
            rates[name].append(n / sec)
    report["windows_per_s"] = rates
    report["median_windows_per_s"] = {k: statistics.median(v) for k, v in rates.items()}
    report["spread_windows_per_s"] = {k: max(v) - min(v) for k, v in rates.items()}
    report["card_after"] = card()
    print(f"{n_eval} evaluated windows ({ev.steps} steps of {args.batch}), {n_inf} record-inference windows")
    for k in names:
        print(f"  {k:18s} median {report['median_windows_per_s'][k]:12.0f} windows/s  "
              f"(spread {report['spread_windows_per_s'][k]:.0f})")
    print("graph == eager (bit for bit):", report["graph_equals_eager"])
    for lv, d in report["fp32_per_level"].items():
        print(f"  fp32 {lv:>5s} dB: n={d['count']} snr_in={d['snr_in']:.4f} snr_out={d['snr_out']:.4f} "
              f"rmse={d['rmse']:.5f}")
    print("card after:", report["card_after"])
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "exp_record_eval.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
