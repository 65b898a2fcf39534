"""TF32 inference precision (inference_precision = "tf32", RL_NET_TF32) against the default fp32 mode.

Speed: the record-inference workload of bench.py --workload infer (48 seeded records x 2 leads x 650000 samples, cut
into 121,872 non-overlapping 256-sample windows, denoise_records(batch=4096)), timed with CUDA events in alternating
rounds of both precisions after a warm-up of each; windows/s per round, median and spread per precision.  Then the
per-kernel table (ralenet_profile_*: one event pair per launch, launches serialised) of one 4096-window batch in each
precision, whose difference shows where the time goes.
Accuracy: the bench records are Gaussian noise without a clean signal, so SNR-mixed synthetic records are used
instead (clean beat trains of synth.py, emb noise at -4 dB): per-record SNR and RMSE of the denoised output against the
clean signal in both precisions, and their difference in dB.
The card name and power limit are read in the same run.

usage: python tools/exp_inference_precision.py [--rounds 3] [--out DIR]
(--out DIR also writes the report to DIR/exp_inference_precision.json)
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

from ecg_denoise_b200 import _lib, inference, synth  # noqa: E402
from ecg_denoise_b200.model import transformer  # noqa: E402
from ecg_denoise_b200.ops import _stream  # noqa: E402
from oracle import ralenet_oracle as O  # noqa: E402

PRECISIONS = ("fp32", "tf32")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return q


def bench_model():
    """the weights of bench.py::bench_state_dict (seed 2023, R-wave tables through parameters_normalize())"""
    torch.manual_seed(2023)
    m = transformer.ralenet(high_level_enhence=True)
    for rw in (m.rwattn1, m.rwattn2, m.rwattn3, m.rwattn4):
        rw.parameters_normalize()
    return m.cuda().eval()


def timed(m, recs, precision, batch):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    inference.denoise_records(m, recs, batch=batch, precision=precision)
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def kernel_table(m, x, precision):
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
    _lib.check(0 if got > 0 else -3)
    table = {}
    for i in range(got):
        lab = labels.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode()
        t = table.setdefault(lab, {"launches": 0, "ms": 0.0})
        t["launches"] += 1
        t["ms"] += float(ms[i])
    return table


def records(R, nwin, tail, seed):
    w = synth.clean_windows(R * (nwin + 1), 2, 256, seed).reshape(R, nwin + 1, 2, 256)
    clean = np.ascontiguousarray(w.transpose(0, 2, 1, 3).reshape(R, 2, (nwin + 1) * 256)[..., :nwin * 256 + tail])
    return torch.from_numpy(synth.add_noise(clean, "emb", -4.0, seed + 1)), torch.from_numpy(clean)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    rep = {"card": card(), "workload": "48 records x 2 leads x 650000 samples -> 121872 windows of 2 x 256, "
                                       f"denoise_records(batch={args.batch})"}
    print("card:", rep["card"])
    m = bench_model()

    # -- speed ---------------------------------------------------------------------------------------------------
    R, T = 48, 650000
    recs = torch.randn(R, 2, T, generator=torch.Generator().manual_seed(100)).cuda()
    nwin = R * inference.windows_per_record(T)
    for p in PRECISIONS:
        timed(m, recs, p, args.batch)                        # warm-up: module load, workspace, smem attributes
    rounds = {p: [] for p in PRECISIONS}
    for r in range(args.rounds):
        for p in (PRECISIONS if r % 2 == 0 else PRECISIONS[::-1]):
            ms = timed(m, recs, p, args.batch)
            rounds[p].append(nwin / (ms * 1e-3))
            print(f"round {r} {p}: {ms:9.2f} ms  {rounds[p][-1]:12.0f} windows/s")
    rep["windows_per_s"] = {p: {"rounds": v, "median": statistics.median(v), "min": min(v), "max": max(v)}
                            for p, v in rounds.items()}
    for p, v in rounds.items():
        print(f"{p}: median {statistics.median(v):.0f} windows/s (min {min(v):.0f}, max {max(v):.0f})")
    speedup = statistics.median(rounds["tf32"]) / statistics.median(rounds["fp32"])
    rep["tf32_over_fp32"] = speedup
    print(f"tf32 / fp32 throughput: {speedup:.3f}")
    del recs

    # -- per-kernel table of one batch ----------------------------------------------------------------------------
    x = torch.randn(args.batch, 2, 256, generator=torch.Generator().manual_seed(1)).cuda()
    tabs = {p: kernel_table(m, x, p) for p in PRECISIONS}
    rep["kernels"] = tabs
    base = lambda lab: lab[:-5] if lab.endswith(":tf32") else lab   # noqa: E731
    rows = {}
    for p, t in tabs.items():
        for lab, v in t.items():
            rows.setdefault(base(lab), {})[p] = v
    print(f"\nper-kernel table, one batch of {args.batch} windows (ms summed over launches)")
    print(f"{'kernel':34s} {'launches':>8s} {'fp32 ms':>9s} {'tf32 ms':>9s} {'delta':>9s}")
    for lab, v in sorted(rows.items(), key=lambda kv: -kv[1].get("fp32", {"ms": 0})["ms"]):
        a, b = v.get("fp32", {"ms": 0.0, "launches": 0}), v.get("tf32", {"ms": 0.0, "launches": 0})
        nl = max(a["launches"], b["launches"])
        print(f"{lab:34s} {nl:8d} {a['ms']:9.3f} {b['ms']:9.3f} {b['ms'] - a['ms']:+9.3f}")
    tot = {p: sum(v["ms"] for v in t.values()) for p, t in tabs.items()}
    print(f"{'total':34s} {'':8s} {tot['fp32']:9.3f} {tot['tf32']:9.3f} {tot['tf32'] - tot['fp32']:+9.3f}")
    rep["kernel_ms_total"] = tot

    # -- accuracy on SNR-mixed synthetic records -------------------------------------------------------------------
    noisy, clean = records(8, 64, 100, 11)
    ys = {p: inference.denoise_records(m, noisy.cuda(), batch=args.batch, precision=p).cpu() for p in PRECISIONS}
    snr = {p: O.SNR(clean, y).numpy() for p, y in ys.items()}
    rmse = {p: O.RMSE(clean, y).numpy() for p, y in ys.items()}
    d_snr = np.abs(snr["tf32"] - snr["fp32"])
    d_rmse = np.abs(20 * np.log10(rmse["tf32"] / rmse["fp32"]))
    print("\nper-record SNR / RMSE against the clean signal (8 records x 2 leads x 16484 samples, emb noise at -4 dB)")
    for i in range(len(d_snr)):
        print(f"record {i}: SNR fp32 {snr['fp32'][i]:9.4f} tf32 {snr['tf32'][i]:9.4f} dB (|d| {d_snr[i]:.2e});  "
              f"RMSE fp32 {rmse['fp32'][i]:.5f} tf32 {rmse['tf32'][i]:.5f} (|d| {d_rmse[i]:.2e} dB)")
    print(f"max |dSNR| {d_snr.max():.2e} dB, max |dRMSE| {d_rmse.max():.2e} dB")
    rep["accuracy"] = {"snr_db": {p: v.tolist() for p, v in snr.items()},
                       "rmse": {p: v.tolist() for p, v in rmse.items()},
                       "max_abs_dsnr_db": float(d_snr.max()), "max_abs_drmse_db": float(d_rmse.max())}
    rep["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "exp_inference_precision.json"), "w") as f:
            json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
