"""Bit-for-bit comparison of two builds of the library on the same seeded inputs (refactors that must not change
arithmetic).

Each run writes the results of one build; --compare then reports, per tensor, whether the two builds agree bit for bit:
  RALENET_B200_LIB=build/variants/base.so python tools/ab_bitwise.py --out DIR/base.npz
  python tools/ab_bitwise.py --out DIR/new.npz
  python tools/ab_bitwise.py --compare DIR/base.npz DIR/new.npz

Cases: the training-mode forward and backward of the whole network (output, dx, every parameter gradient) at B = 256
and 515, in the default and the deterministic mode; the no-grad forward in fp32 and TF32 at the same batches.  Each
case runs with the attention forward chosen by the default rule and with the tcgen05 tile kernels forced on
(ralenet_set_attn_umma(2)).  The default mode adds weight gradients with float atomics, so each of its cases runs twice
and a tensor that already differs between two runs of one build is reported as such, not as a mismatch.
"""
from __future__ import annotations

import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def model():
    from ecg_denoise_b200.model import transformer
    from oracle import synth_weights as SW
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(SW.make_state_dict("rw", 1, 2023), strict=True)
    return m.cuda()


def batch(B: int) -> torch.Tensor:
    from ecg_denoise_b200 import synth
    noisy, _ = synth.make_batch(B, 2, 256, seed=B)
    return torch.from_numpy(noisy).cuda()


def train_case(m, x, det: bool) -> dict:
    m.train()
    m.zero_grad(set_to_none=True)
    xr = x.clone().requires_grad_(True)
    torch.use_deterministic_algorithms(det)
    try:
        y = m(xr)
        g = torch.Generator(device="cpu").manual_seed(7)
        (y * torch.randn(y.shape, generator=g).cuda()).sum().backward()
    finally:
        torch.use_deterministic_algorithms(False)
    out = {"y": y, "dx": xr.grad}
    out.update({"grad." + k: p.grad for k, p in m.named_parameters() if p.grad is not None})
    return {k: v.detach().cpu().numpy().copy() for k, v in out.items()}


def infer_case(m, x, precision: str) -> dict:
    m.eval()
    m.inference_precision = precision
    try:
        with torch.no_grad():
            y = m(x)
    finally:
        m.inference_precision = "fp32"
    return {"y": y.cpu().numpy().copy()}


def run(out_path: str) -> None:
    from ecg_denoise_b200 import _lib
    res = {}
    for umma in ("default", "forced"):
        prev = _lib.set_attn_umma(2) if umma == "forced" else None
        try:
            for B in (256, 515):
                x = batch(B)
                for det in (False, True):
                    name = f"train/{'det' if det else 'fp32'}/B{B}/{umma}"
                    for rep in range(1 if det else 2):
                        m = model()
                        for k, v in train_case(m, x, det).items():
                            res[f"{name}/run{rep}/{k}"] = v
                for prec in ("fp32", "tf32"):
                    for k, v in infer_case(model(), x, prec).items():
                        res[f"infer/{prec}/B{B}/{umma}/run0/{k}"] = v
        finally:
            if prev is not None:
                _lib.set_attn_umma(prev)
    np.savez(out_path, **res)
    print(f"{len(res)} tensors -> {out_path}")


def compare(a_path: str, b_path: str) -> int:
    a, b = np.load(a_path), np.load(b_path)
    assert set(a.files) == set(b.files), "the two runs hold different cases"
    same = differ = noisy = 0
    for k in sorted(a.files):
        if "/run1/" in k:
            continue
        va, vb = a[k], b[k]
        if va.tobytes() == vb.tobytes():
            same += 1
            continue
        k1 = k.replace("/run0/", "/run1/")
        if k1 in a.files and a[k].tobytes() != a[k1].tobytes():
            noisy += 1          # not reproducible within one build either
            continue
        differ += 1
        print(f"DIFFERS {k}: max |a - b| = {np.abs(va.astype(np.float64) - vb).max():.3e}")
    print(f"bit-identical {same}, differ {differ}, not reproducible within a build {noisy}")
    return 1 if differ else 0


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        return compare(*args.compare)
    run(args.out)
    return 0


if __name__ == "__main__":
    sys.exit(main())
