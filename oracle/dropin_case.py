"""The drop-in driver case: the reference's own `denoise_train.train` (denoise_train.py:14-103, UNCHANGED, imported
from the reference root) driven for 2 epochs on synthetic loaders.  TEST INFRASTRUCTURE ONLY.

Used twice: by `oracle/make_golden_dropin.py` with the reference's model on the CPU (-> tests/golden/dropin_golden.json)
and by `tests/test_dropin_driver.py` with `ecg_denoise_b200.install()` on the B200.  `global_utils` (un-vendored by the
reference) comes from the test-only shim in tests/shim/.  `stock_train` restates the same loop so that the numbers of
the golden file are also checked where the reference is not at hand.
"""
from __future__ import annotations

import contextlib
import importlib
import io
import os
import sys
import tempfile

import numpy as np
import torch
from torch.utils.data import DataLoader, TensorDataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "tests", "shim")
EPOCHS, BATCH, N_TRAIN, N_TEST = 2, 16, 64, 32


def loaders():
    from ecg_denoise_b200 import synth
    noisy, clean = synth.make_batch(N_TRAIN + N_TEST, 2, 256, seed=4242, kind="bw", snr_db=-4.0)
    x, t = torch.from_numpy(noisy), torch.from_numpy(clean)
    tr = DataLoader(TensorDataset(x[:N_TRAIN], t[:N_TRAIN]), BATCH, shuffle=False)
    te = DataLoader(TensorDataset(x[N_TRAIN:], t[N_TRAIN:]), BATCH, shuffle=False)
    return tr, te


def import_denoise_train(ref_root: str):
    """`import denoise_train` exactly as main.py:61 does, from the reference root, with the shim for global_utils."""
    for p in (SHIM, ref_root):
        if p not in sys.path:
            sys.path.insert(0, p)
    sys.modules.pop("denoise_train", None)
    return importlib.import_module("denoise_train")


def run_train(ref_root: str, model, use_gpu: bool):
    """returns (train_snr_list, test_snr_list, train_rmse_list, test_rmse_list) of denoise_train.train."""
    dt = import_denoise_train(ref_root)
    tr, te = loaders()
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as d:
        os.chdir(d)                      # train() appends to ./output.txt
        try:
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                res = dt.train(epochs=EPOCHS, model=model, batch_size=BATCH, train_loader=tr, test_loader=te,
                               use_gpu=use_gpu, model_name="ralenet", noise_name="bw", noise_intensity=-4)
            line = open("output.txt").read().strip()
        finally:
            os.chdir(cwd)
    return [list(map(float, r)) for r in res], line


def stock_train(model):
    """the loop of denoise_train.train on the GPU, restated: model.cuda(), Adam(lr 1e-3); every epoch, train mode over
    the training batches (zero_grad, model(data), F.mse_loss, loss.item(), backward, step, per-window SNR / RMSE of
    that output), then eval mode over the test batches (without torch.no_grad, as the reference runs it).  Returns
    (train_snr, test_snr, train_rmse, test_rmse), each the per-epoch mean over windows, like run_train."""
    import torch.nn.functional as F
    from oracle.ralenet_oracle import RMSE, SNR
    tr, te = loaders()
    model = model.cuda()
    opt = torch.optim.Adam(model.parameters(), lr=0.001)

    def metrics(target, pre):
        t, p = target.double(), pre.detach().cpu().double()
        return SNR(t, p), RMSE(t, p)

    res = [[], [], [], []]
    for _ in range(EPOCHS):
        model.train()
        snr, rmse = [], []
        for data, target in tr:
            opt.zero_grad()
            pre = model(data.cuda())
            loss = F.mse_loss(pre, target.cuda())
            loss.item()
            loss.backward()
            opt.step()
            s, r = metrics(target, pre)
            snr.append(s)
            rmse.append(r)
        res[0].append(float(torch.cat(snr).mean()))
        res[2].append(float(torch.cat(rmse).mean()))
        model.eval()
        snr, rmse = [], []
        for data, target in te:
            s, r = metrics(target, model(data.cuda()))
            snr.append(s)
            rmse.append(r)
        res[1].append(float(torch.cat(snr).mean()))
        res[3].append(float(torch.cat(rmse).mean()))
    return res
