#!/usr/bin/env python
"""bench.py -- RA-LENet training-step throughput on B200 (BASELINE.json metric: ECG windows/s).

    python bench.py --gpus N --steps K --warmup W            # one rank per GPU under torchrun for N > 1
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy
    python bench.py --impl reference ...                     # the UNMODIFIED reference on this box's host cores
    python bench.py --impl reference-gpu ...                 # the UNMODIFIED reference, eager PyTorch, on the B200

Headline workload (SURVEY.md section 8d): BASELINE.json configs[1] "RA-LENet single-lead training step (fwd+bwd+Adam),
batch 256 x 1 x 512" realised reference-natively as 256 windows of 2 x 256 samples (the reference's conv1 is
hard-wired to 2 leads x 256 samples, SURVEY F1), model = transformer.ralenet(high_level_enhence=True), MSE loss,
Adam lr 1e-3, fp32.  One "step" = forward + loss + backward + (gradient all-reduce) + Adam on one batch of
synthetic windows.  N > 1: `value` is weak scaling, 256 windows per GPU (so that N = 1 is the BENCH line), BatchNorm
statistics and the flat gradient buffer all-reduced (equals the single-process step on the global batch).

Prints ONE JSON line (rank 0).  `value` = windows/s with inputs resident in HBM, CUDA-event timed, max over
ranks; `e2e` = the same through FusedTrainer.step_host with pinned HOST buffers (H2D of the batch and D2H of the
loss inside the timed region); `roofline` = the dominant kernel, timed live per launch with CUDA events
(ralenet_profile_*); `cpu_baseline` = the reference's own modules (baseline/_ref) on this box's host cores.
Sub-records of the same line (each the north star's other configs, measured in the same run):
  config4            configs[3]: data-parallel training at GLOBAL batch 4096 (4096/N windows per GPU; N = 1: one GPU
                     at 4096) -- strong scaling
  dp_parity          N > 1: after 3 steps the data-parallel model equals the single-process model on the global batch
  inference          configs[4]: 48 records x 650000 samples -> 121,872 windows, sharded by record, no communication
  config3            configs[2]: 12-lead fine-tune step (newrale, frozen core) at 1280 windows of 12 x 256
  dropin             the stock loop of denoise_train.py:51-57 (model(data), F.mse_loss, .item(), backward,
                     torch.optim.Adam) through the drop-in nn.Module -- the cost of NOT adopting FusedTrainer
  eager_gpu_baseline the unmodified reference modules, eager PyTorch, on the same B200 (fp32 and TF32)
  whole_step         algorithmic FLOP/s and HBM B/s of the whole step against the measured peaks
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "RA-LENet train-step throughput (fwd+bwd+Adam)"
UNIT = "windows/s"
PER_GPU_BATCH = 256
GLOBAL_BATCH_CONFIG4 = 4096
WORKLOAD = ("configs[1]: RA-LENet training step (fwd+bwd+Adam, MSE, lr 1e-3), {b} windows x 2 leads x 256 samples "
            "per GPU (= 256 x 1 x 512 samples; reference-native shape, SURVEY F1), transformer.ralenet("
            "high_level_enhence=True), fp32")
FLOPS_PER_WINDOW_TRAIN = 184_665_984       # torch.utils.flop_counter on the reference, SURVEY 8d
BYTES_PER_WINDOW_TRAIN = 2_347_008         # fp32 activations, per-half-block schedule, SURVEY 8d
ADAM_BYTES_PER_STEP = 7 * 4 * 1_087_282
# --dump-outputs writes at most this many windows (32 MiB of `out`), so that a dump stays under 64 MB with the model state
DUMP_MAX_WINDOWS = 16384


def workload_config(world: int, B: int, graph: bool = True):
    """the `config` object -- identical for this arm and the reference arms (same workload)."""
    return {"workload": WORKLOAD.format(b=B), "global_batch": world * B,
            "parallelism": f"dp{world}" if world > 1 else "single",
            "l2": "no explicit flush: each step streams 466 MB of saved activations (> 126 MB L2) and "
                  "rotates over 4 different input batches"}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        return {}


# ------------------------------------------------------------------------------------------------------
def algorithmic_work(label: str, B: int, L0: int = 256):
    """(flops, bytes) per launch of a kernel label 'name<C>': 2*MAC of the matmul-shaped work only, and the fp32
    activation tensors that algorithmically cross HBM in a TRAINING step (block input/output plus the tensors saved
    for / read by the backward: q,k,v,o,lse = 4.25 N and the fc1 pre-activation = 4 N; DESIGN.md section 4)."""
    name, _, tag = label.partition("<")
    tags = [int(t) for t in tag.rstrip(">").split(",") if t.strip().lstrip("-").isdigit()] if tag else []
    N = 8 * L0                       # floats per window per activation tensor
    alias = {"ffn_fwd_cluster": "ffn_fwd_kernel", "ffn_bwd_cluster": "ffn_bwd_kernel",
             "ffn_fwd_umma": "ffn_fwd_kernel", "ffn_bwd_umma": "ffn_bwd_kernel",
             "attn_fwd_umma": "attn_fwd_kernel", "attn_bwd_umma": "attn_bwd_kernel"}
    name = alias.get(name, name)
    if name == "block_fwd_kernel" and tags:       # fused attention + feed-forward half (narrow stages): x in, x1 and y
        C = tags[0]                                # out, q,k,v,o,lse (4.25 N) and h (4 N) saved
        L = N // C
        return B * (8 * L * C * C + 4 * L * L * C + 16 * L * C * C), int(B * 11.25 * N * 4)
    if name in ("attn_fwd_kernel", "attn_bwd_kernel", "ffn_fwd_kernel", "ffn_bwd_kernel") and tags:
        C = tags[0]
        L = N // C
        if name == "attn_fwd_kernel":
            return B * (8 * L * C * C + 4 * L * L * C), int(B * 6.25 * N * 4)
        if name == "attn_bwd_kernel":
            return B * (8 * L * C * C + 8 * L * L * C), int(B * 7.25 * N * 4)
        if name == "ffn_fwd_kernel":
            return B * 16 * L * C * C, B * 6 * N * 4
        return B * 16 * L * C * C, B * 7 * N * 4
    if name in ("patch_fwd_kernel", "patch_bwd_kernel") and tags:
        CN = tags[0]
        rows = N // CN
        return B * 2 * rows * CN * CN, B * (3 if name == "patch_fwd_kernel" else 4) * N * 4
    return 0, None


def sample_clocks(stop_evt, path):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                             stdout=open(path, "w"), stderr=subprocess.DEVNULL)
    except OSError:
        return
    stop_evt.wait()
    p.terminate()
    try:
        p.wait(timeout=5)
    except Exception:
        p.kill()


def parse_clocks(path, gpu_index):
    sm, mx, reasons = [], [], set()
    try:
        for line in open(path):
            f = [t.strip() for t in line.split(",")]
            if len(f) < 9 or f[0] != str(gpu_index):
                continue
            sm.append(float(f[1])); mx.append(float(f[2]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
    except OSError:
        pass
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    busy = sorted(sm)[len(sm) // 2:]          # upper half = samples under load
    return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# baselines: the reference's own code (baseline/_ref, mirrored from /root/reference by oracle/build_ref.py)
def bench_state_dict():
    """the benchmark weights: random init of the benchmark architecture under seed 2023 (main.py:24), R-wave tables
    randomised with the reference's own parameters_normalize() so the bias path does real work.  Built from the
    module mirror on the CPU (constructors only -- no kernel is involved) so both arms start from identical weights."""
    import torch
    from ecg_denoise_b200.model import transformer
    torch.manual_seed(2023)
    model = transformer.ralenet(high_level_enhence=True)
    for rw in (model.rwattn1, model.rwattn2, model.rwattn3, model.rwattn4):
        rw.parameters_normalize()
    return model, {k: v.clone() for k, v in model.state_dict().items()}


def reference_model(sd):
    """transformer.ralenet(high_level_enhence=True) of the UNMODIFIED reference with the benchmark weights, or None."""
    from oracle import ref_loader
    R = ref_loader.load_reference()
    if R is None:
        return None, None
    m = R.quiet(R.transformer.ralenet, high_level_enhence=True)
    m.load_state_dict(sd, strict=True)
    return m, R


def reference_train_loop(model, x, t, lr=1e-3, opt=None):
    """denoise_train.py:24, 51-57 verbatim in behaviour: Adam(lr 1e-3); zero_grad, model(data), F.mse_loss,
    loss.item(), backward, step.  (`opt`: another optimizer object for the same loop.)"""
    import torch
    import torch.nn.functional as F
    if opt is None:
        opt = torch.optim.Adam(model.parameters(), lr=lr)
    model.train()

    def step():
        opt.zero_grad()
        pre = model(x)
        loss = F.mse_loss(pre, t)
        v = loss.item()
        loss.backward()
        opt.step()
        return v
    return step


def cpu_port_step_factory(B, threads):
    """fallback when baseline/_ref is absent: the oracle port (fwd, MSE, manual bwd, Adam on every tensor)."""
    import torch
    from ecg_denoise_b200 import synth
    from oracle import ralenet_oracle as O
    from oracle import synth_weights as SW
    torch.set_num_threads(threads)
    sd = SW.make_state_dict("rw", 1, 2023)
    noisy, clean = synth.make_batch(B, 2, 256, seed=2023)
    x, t = torch.from_numpy(noisy), torch.from_numpy(clean)
    names = O.trainable_keys(sd)
    m = {n: torch.zeros_like(sd[n]) for n in names}
    v = {n: torch.zeros_like(sd[n]) for n in names}
    state = {"step": 0}

    def step():
        state["step"] += 1
        with torch.no_grad():
            out, ctx, new_stats = O.ralenet_fwd(x, sd, training=True)
            loss, dout = O.mse_loss_fwd_bwd(out, t)
            _, grads = O.ralenet_bwd(dout, ctx, sd)
            for n in names:
                O.adam_step(sd[n], grads[n], m[n], v[n], state["step"])
            sd["conv1.2.running_mean"], sd["conv1.2.running_var"] = new_stats[0], new_stats[1]
        return float(loss)
    return step


def cpu_reference_step(B):
    """(step fn, kind, threads): the reference's CPU training step on B windows, all host threads."""
    import torch
    from ecg_denoise_b200 import synth
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    _, sd = bench_state_dict()
    model, _ = reference_model(sd)
    if model is None:
        return cpu_port_step_factory(B, threads), "port", threads
    noisy, clean = synth.make_batch(B, 2, 256, seed=2023)
    return reference_train_loop(model, torch.from_numpy(noisy), torch.from_numpy(clean)), "reference", threads


def time_cpu_baseline(budget_s=12.0, B=PER_GPU_BATCH):
    step, kind, threads = cpu_reference_step(B)
    step()
    n, t0 = 0, time.perf_counter()
    while True:
        step()
        n += 1
        el = time.perf_counter() - t0
        if el >= budget_s or n >= 200:
            break
    what = ("the unmodified reference (baseline/_ref: transformer.ralenet + autograd + torch.optim.Adam)"
            if kind == "reference" else "the oracle port (baseline/_ref absent)")
    return {"value": n * B / el, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{n} train steps (fwd+bwd+Adam) of {what} on {B} x 2 x 256 windows, "
                      f"{el:.1f} s, torch CPU fp32, {threads} threads"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (unmodified modules from baseline/_ref,
    autograd, torch.optim.Adam) on all host threads, on this arm's config: 256 windows per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = PER_GPU_BATCH
    step, kind, threads = cpu_reference_step(B)
    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    el = time.perf_counter() - t0
    val = args.steps * B / el
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1, B),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"{args.steps} train steps of "
                                   + ("the unmodified reference (baseline/_ref)" if kind == "reference"
                                      else "the oracle port") + f" on {B} x 2 x 256 windows, {threads} threads"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def time_eager_gpu(dev, sd, B, steps, warmup, tf32: bool):
    """the unmodified reference modules, eager PyTorch on the GPU, denoise_train.py's loop.  windows/s or None."""
    import torch
    from ecg_denoise_b200 import synth
    model, _ = reference_model(sd)
    if model is None:
        return None
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.backends.cudnn.allow_tf32 = tf32
    try:
        model = model.to(dev)
        noisy, clean = synth.make_batch(B, 2, 256, seed=2023)
        x, t = torch.from_numpy(noisy).to(dev), torch.from_numpy(clean).to(dev)
        step = reference_train_loop(model, x, t)
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))
        return {"value": B * steps / (ms * 1e-3), "ms_per_step": ms / steps}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def eager_gpu_baseline(dev, sd, B, steps=10, warmup=3):
    a = time_eager_gpu(dev, sd, B, steps, warmup, tf32=False)
    if a is None:
        return {"unavailable": "baseline/_ref absent (run python -m oracle.build_ref where /root/reference exists)"}
    b = time_eager_gpu(dev, sd, B, steps, warmup, tf32=True)
    return {"value": a["value"], "unit": UNIT, "ms_per_step": a["ms_per_step"], "dtype": "f32",
            "tf32": {"value": b["value"], "ms_per_step": b["ms_per_step"]},
            "what": f"unmodified reference transformer.ralenet(high_level_enhence=True), eager PyTorch on the same "
                    f"B200, denoise_train.py:51-57 loop (autograd, torch.optim.Adam, loss.item()), {B} x 2 x 256 "
                    f"windows, {steps} steps after {warmup} warm-up"}


def run_reference_gpu(args):
    """--impl reference-gpu: the same-box bar SURVEY 2.2 / 8d names -- the reference, eager, on the B200."""
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device("cuda", 0)
    _, sd = bench_state_dict()
    r = time_eager_gpu(dev, sd, PER_GPU_BATCH, args.steps, args.warmup, tf32=False)
    if r is None:
        print(json.dumps({"impl": "reference-gpu", "unavailable": "baseline/_ref absent"}))
        return
    print(json.dumps({
        "impl": "reference-gpu", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1, PER_GPU_BATCH)}))


# ------------------------------------------------------------------------------------------------------
def dist_env():
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    return world, rank, local_rank, torch.device("cuda", local_rank)


def max_over_ranks(vals, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor(vals, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def inference_record(model, dev, world, rank, steps, warmup):
    """configs[4]: batch-sharded inference on 48 synthetic 650000-sample 2-lead records (30 min @ 360 Hz) cut into
    non-overlapping 256-sample windows (the reference's cut, local_utils/local_utils.py:53): 2539 windows per record,
    121,872 in total, sharded by record across ranks with no communication.  One step = all records of this rank:
    z-norm + window gather, eval forward, stitch."""
    import torch
    import torch.distributed as dist
    from ecg_denoise_b200 import inference
    R_total, T = 48, 650000
    R = R_total // world
    was_training = model.training
    model.eval()
    g = torch.Generator().manual_seed(100 + rank)
    host = torch.randn(R, 2, T, generator=g).pin_memory()
    recs = host.to(dev)
    nper = inference.windows_per_record(T)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 1)):
        y = inference.denoise_records(model, recs, batch=4096)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        y = inference.denoise_records(model, recs, batch=4096)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    out_host = torch.empty_like(host).pin_memory()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        recs.copy_(host, non_blocking=True)
        y = inference.denoise_records(model, recs, batch=4096)
        out_host.copy_(y, non_blocking=True)
        torch.cuda.synchronize()
    ms_e2e = 1e3 * (time.perf_counter() - t0)
    ms, ms_e2e = max_over_ranks([ms, ms_e2e], dev, world)
    model.train(was_training)
    del recs, y, host, out_host
    nwin = world * R * nper
    return {"metric": "RA-LENet inference throughput (records -> windows -> denoise -> stitch)",
            "value": nwin * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "scaling": "strong",
            "steps": steps,
            "workload": f"configs[4]: {world * R} records x 2 leads x {T} samples -> {nwin} windows of 2 x 256, "
                        "eval forward (no_grad: no activations saved), batch-sharded by record, no communication",
            "e2e": {"value": nwin * steps / (ms_e2e * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": R * 2 * T * 4, "d2h_bytes_per_step": R * 2 * T * 4}}


def run_inference(args):
    import torch
    import torch.distributed as dist
    world, rank, local_rank, dev = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model, _ = bench_state_dict()
    model = model.to(dev)
    rec = inference_record(model, dev, world, rank, args.steps, args.warmup)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        rec.update({"n_gpus": world, "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic", "config": {"workload": rec.pop("workload")}})
        print(json.dumps(rec))


def train12_record(dev, world, rank, steps, warmup):
    """configs[2]: 12-lead fine-tuning step (ralenet_12leads.newrale: 4 x Conv1d k13 around the frozen RA-LENet
    core, Transfer_learning.py:71-75).  64 LUDB-shaped records x 12 leads x 5000 samples per GPU, zero-padded to
    5120 and cut into 20 windows of 256 -> 1280 windows of 12 x 256 per step; MSE, torch.optim.Adam(lr 1e-3) over
    the 2,210 trainable parameters, through the drop-in nn.Module API (autograd nodes -> C ABI)."""
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    from ecg_denoise_b200 import _lib
    from ecg_denoise_b200.model import ralenet_12leads
    torch.manual_seed(2023)
    core = ralenet_12leads.ralenet(high_level_enhence=True)
    for rw in (core.rwattn1, core.rwattn2, core.rwattn3, core.rwattn4):
        rw.parameters_normalize()
    model = ralenet_12leads.newrale(core).to(dev).train()
    if world > 1:       # SyncBN-equivalent statistics of the core's stem, as in the single-lead path
        core._plan.reduce_fn = lambda t: dist.all_reduce(t)
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=1e-3)
    R, T, NW = 64, 5000, 20
    g = torch.Generator().manual_seed(300 + rank)
    rec = torch.zeros(2, R, 12, NW * 256)
    rec[..., :T] = torch.randn(2, R, 12, T, generator=g)
    # (R, 12, 5120) -> (R * 20, 12, 256) windows
    hwin = rec.view(2, R, 12, NW, 256).permute(0, 1, 3, 2, 4).reshape(2, R * NW, 12, 256).contiguous().pin_memory()
    hx, ht = hwin[0], hwin[1]
    dx, dt = hx.to(dev), ht.to(dev)
    B = R * NW

    def step(x, t):
        opt.zero_grad(set_to_none=True)
        loss = F.mse_loss(model(x), t)
        loss.backward()
        if world > 1:
            for p in params:
                dist.all_reduce(p.grad)
                p.grad.div_(world)
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step(dx, dt)
    barrier()
    _lib.launch_count(reset=True)
    step(dx, dt)
    torch.cuda.synchronize()
    launches = _lib.launch_count(reset=True)
    # the stock loop allocates through the caching allocator every step (a 2.3 GB workspace lease among others), so a
    # timed loop right after other large workloads can include one-off cudaMalloc / cudaFree stalls: best of two loops
    ms = float("inf")
    for _ in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            loss = step(dx, dt)
        e1.record()
        barrier()
        ms = min(ms, e0.elapsed_time(e1))
    sx, st_ = torch.empty_like(dx), torch.empty_like(dt)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        sx.copy_(hx, non_blocking=True)
        st_.copy_(ht, non_blocking=True)
        host_loss = step(sx, st_).item()
    barrier()
    ms_e2e = 1e3 * (time.perf_counter() - t0)
    ms, ms_e2e = max_over_ranks([ms, ms_e2e], dev, world)
    fused = None
    if world == 1:
        # the same step through engine.FineTuneTrainer: C ABI calls on static buffers, flat Adam, ONE CUDA graph
        from ecg_denoise_b200.engine import FineTuneTrainer
        ft = FineTuneTrainer(model, lr=1e-3, use_graph=True)
        for _ in range(warmup):
            ft.step(dx, dt)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(steps):
            ft.step(dx, dt)
        f1.record()
        torch.cuda.synchronize()
        fms = f0.elapsed_time(f1)
        ft.prefetch_host(hx, ht)                   # (warm-up of the pipelined loop: staging pair, copy stream, slots)
        ft.read_async(ft.step_host(hx, ht))()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ft.prefetch_host(hx, ht)
        pend = []
        for _ in range(steps):                    # same software pipeline as the main e2e loop (see main())
            pend.append(ft.read_async(ft.step_host(hx, ht)))
            ft.prefetch_host(hx, ht)
            if len(pend) > 2:
                fl = pend.pop(0)()
        while pend:
            fl = pend.pop(0)()
        torch.cuda.synchronize()
        fms_e2e = 1e3 * (time.perf_counter() - t0)
        fused = {"value": B * steps / (fms * 1e-3), "unit": "12-lead windows/s", "ms_per_step": fms / steps,
                 "e2e": {"value": B * steps / (fms_e2e * 1e-3), "unit": "12-lead windows/s",
                         "h2d_bytes_per_step": 2 * B * 12 * 256 * 4, "d2h_bytes_per_step": 4},
                 "final_loss": float(fl),
                 "what": "engine.FineTuneTrainer: the same kernels through the C ABI on static buffers, flat Adam, "
                         "whole step replayed from one CUDA graph"}
        ft.close()
    return {"metric": "RA-LENet 12-lead fine-tune step throughput (fwd+bwd+Adam, frozen core)",
            "value": world * B * steps / (ms * 1e-3), "unit": "12-lead windows/s", "ms_per_step": ms / steps,
            "steps": steps, "scaling": "weak", "fused_graph": fused,
            "workload": f"configs[2]: newrale(ralenet(high_level_enhence=True)), {R} records x 12 x {T} per GPU "
                        f"-> {B} windows of 12 x 256 per step (reference-native shape, SURVEY F2), MSE, "
                        "torch.optim.Adam lr 1e-3 on the 4 Conv1d k13 layers, core frozen",
            "global_batch": world * B,
            "e2e": {"value": world * B * steps / (ms_e2e * 1e-3), "unit": "12-lead windows/s",
                    "h2d_bytes_per_step": 2 * B * 12 * 256 * 4, "d2h_bytes_per_step": 4},
            "launches_per_step": launches, "final_loss": float(host_loss)}


def run_train12(args):
    import torch.distributed as dist
    world, rank, local_rank, dev = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rec = train12_record(dev, world, rank, args.steps, args.warmup)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        rec.update({"n_gpus": world, "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic",
                    "config": {"workload": rec.pop("workload"), "global_batch": rec.pop("global_batch"),
                               "parallelism": f"dp{world}" if world > 1 else "single"},
                    "gpu_launches": rec["launches_per_step"] * args.steps})
        print(json.dumps(rec))


def dropin_record(dev, sd, B, steps, warmup):
    """the stock training loop of denoise_train.py:24, 51-57 on the drop-in module (one autograd node per forward,
    torch.optim.Adam over the ~300 parameter tensors, loss.item() every step)."""
    import torch
    from ecg_denoise_b200 import _lib, synth
    from ecg_denoise_b200.model import transformer
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(sd)
    m = m.to(dev)
    noisy, clean = synth.make_batch(B, 2, 256, seed=2023)
    x, t = torch.from_numpy(noisy).to(dev), torch.from_numpy(clean).to(dev)
    step = reference_train_loop(m, x, t)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    _lib.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))
    own = _lib.launch_count(reset=True) // steps
    # the same loop with ONE line changed: the optimizer is ecg_denoise_b200.optim.Adam (one kernel over the flat
    # parameter buffer instead of torch's foreach pass over ~300 tensors)
    from ecg_denoise_b200 import optim as rl_optim
    m2 = transformer.ralenet(high_level_enhence=True)
    m2.load_state_dict(sd)
    m2 = m2.to(dev)
    step2 = reference_train_loop(m2, x, t, opt=rl_optim.Adam(m2, lr=1e-3))
    for _ in range(warmup):
        step2()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss2 = step2()
    torch.cuda.synchronize()
    ms2 = 1e3 * (time.perf_counter() - t0)
    return {"value": B * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
            "final_loss": float(loss), "own_launches_per_step": own,
            "what": f"denoise_train.py:51-57 loop on ecg_denoise_b200.model.transformer.ralenet: zero_grad, model(data), "
                    f"F.mse_loss, loss.item(), backward, torch.optim.Adam.step; {B} x 2 x 256 windows",
            "flat_adam": {"value": B * steps / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2 / steps,
                          "final_loss": float(loss2),
                          "what": "the same loop, optimizer line changed to ecg_denoise_b200.optim.Adam(model, lr=1e-3)"}}


def dump_outputs(path, loss, rmse, snr, out, model):
    """--dump-outputs: what the last timed step returned (loss, per-window RMSE and SNR, the denoised windows) and the
    model state it left (every floating-point state_dict tensor, flattened and concatenated in state_dict order), as
    <path>/<name>.npy.  Above DUMP_MAX_WINDOWS windows, the same seeded sample of windows is written every run."""
    import numpy as np
    import torch
    arrays = {"loss": loss, "rmse": rmse, "snr": snr, "out": out}
    if out.shape[0] > DUMP_MAX_WINDOWS:
        idx = np.sort(np.random.default_rng(0).choice(out.shape[0], DUMP_MAX_WINDOWS, replace=False))
        idx = torch.from_numpy(idx).to(out.device)
        arrays.update({k: arrays[k].index_select(0, idx) for k in ("rmse", "snr", "out")})
    arrays["model_state"] = torch.cat([t.detach().reshape(-1) for t in model.state_dict().values()
                                       if t.is_floating_point()])
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().cpu().numpy())


def timed_train(trainer, dx, dt, steps, warmup, barrier):
    import torch
    NB = dx.shape[0]
    for i in range(warmup):
        trainer.step(dx[i % NB], dt[i % NB])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        res = trainer.step(dx[i % NB], dt[i % NB])
    e1.record()
    barrier()
    return e0.elapsed_time(e1), res


def config4_record(dev, sd, world, rank, steps, warmup, barrier):
    """configs[3]: data-parallel training at global batch 4096 x 2 x 256 (4096 / N windows per GPU), SyncBN-equivalent
    statistics + one gradient all-reduce; strong scaling (the global batch is fixed)."""
    import torch
    from ecg_denoise_b200 import synth
    from ecg_denoise_b200.engine import FusedTrainer
    from ecg_denoise_b200.model import transformer
    Bg = GLOBAL_BATCH_CONFIG4
    Bl = Bg // world
    m = transformer.ralenet(high_level_enhence=True)
    m.load_state_dict(sd)
    m = m.to(dev)
    noisy, clean = synth.make_batch(Bl, 2, 256, seed=4096 + 31 * rank)
    x, t = torch.from_numpy(noisy).to(dev), torch.from_numpy(clean).to(dev)
    dx = torch.stack([x, x.flip(0)])            # two different batch orders, rotated
    dt = torch.stack([t, t.flip(0)])
    tr = FusedTrainer(m, lr=1e-3, use_graph=True)
    ms, res = timed_train(tr, dx, dt, steps, warmup, barrier)
    ms, = max_over_ranks([ms], dev, world)
    loss = float(res[0].item())
    tr.close()
    del tr, dx, dt, m
    torch.cuda.empty_cache()
    return {"global_batch": Bg, "per_gpu_batch": Bl, "value": Bg * steps / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms / steps, "steps": steps, "scaling": "strong", "final_loss": loss,
            "what": "configs[3]: FusedTrainer step (CUDA graph, collectives inside) at global batch 4096 x 2 x 256"}


def dp_parity_record(dev, sd, world, rank):
    """after 3 steps from identical weights, the data-parallel model (each rank its slice of ONE global batch) must
    equal the single-process model trained on the whole batch: max relative error over all parameters (tolerance
    definition of BASELINE.md section 3), BatchNorm running statistics and the losses."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from ecg_denoise_b200 import synth
    from ecg_denoise_b200.engine import FusedTrainer
    from ecg_denoise_b200.model import transformer
    Bg = 128 * world
    noisy, clean = synth.make_batch(Bg, 2, 256, seed=777)

    def run(x, t, single):
        m = transformer.ralenet(high_level_enhence=True)
        m.load_state_dict(sd)
        m = m.to(dev)
        tr = FusedTrainer(m, lr=1e-3, use_graph=True)
        if single:
            tr.world = 1
        losses = []
        for _ in range(3):
            losses.append(float(tr.step(x, t)[0].item()))
        tr.close()
        return m, losses

    lo, hi = rank * Bg // world, (rank + 1) * Bg // world
    m_dp, l_dp = run(torch.from_numpy(noisy[lo:hi]).to(dev), torch.from_numpy(clean[lo:hi]).to(dev), False)
    rec = None
    if rank == 0:
        m_1, l_1 = run(torch.from_numpy(noisy).to(dev), torch.from_numpy(clean).to(dev), True)
        worst, worst_name, kvb = 0.0, "", 0.0
        for (n, p), (_, q) in zip(m_dp.named_parameters(), m_1.named_parameters()):
            a, b = p.detach().double().cpu().numpy(), q.detach().double().cpu().numpy()
            if n.endswith("to_kv.bias"):
                # key half: exact gradient is zero (softmax is shift invariant), Adam normalises rounding noise --
                # not a comparable quantity; the value half is compared
                C = a.size // 2
                a, b = a[C:], b[C:]
            e = float(np.max(np.abs(a - b) / (np.abs(b) + np.sqrt((b * b).mean()) + 1e-30)))
            if e > worst:
                worst, worst_name = e, n
        bn_d, bn_1 = m_dp.conv1[2], m_1.conv1[2]
        e_bn = max(float((bn_d.running_var - bn_1.running_var).abs().max()),
                   float((bn_d.running_mean - bn_1.running_mean).abs().max()))
        e_loss = max(abs(a - b) / abs(b) for a, b in zip(l_dp, l_1))
        rec = {"max_rel_err_params": worst, "worst_param": worst_name, "bn_running_stats_abs_err": e_bn,
               "loss_rel_err": e_loss, "steps": 3, "global_batch": Bg, "tolerance": 1e-3,
               "ok": bool(worst < 1e-3 and e_bn < 1e-5 and e_loss < 1e-4)}
    dist.barrier()
    return rec


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="windows per GPU")
    ap.add_argument("--graph", default="on", choices=["on", "off"], help="replay the step from a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the sub-records (config4, dp_parity, inference, config3, dropin, eager_gpu_baseline)")
    ap.add_argument("--dump-kernels", default=None, help="write the per-kernel timing table (JSON) here")
    ap.add_argument("--workload", default="train", choices=["train", "infer", "train12"],
                    help="train = configs[1] (default, the headline); infer = configs[4] record inference; "
                         "train12 = configs[2] 12-lead fine-tuning")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed (loss, rmse, snr, out, model_state) "
                         "as DIR/<name>.npy; the inputs depend only on the arguments, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "train"):
        ap.error("--dump-outputs applies to the default training workload (--impl b200 --workload train)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "reference-gpu":
        return run_reference_gpu(args)
    if args.workload == "infer":
        return run_inference(args)
    if args.workload == "train12":
        return run_train12(args)

    import torch
    import torch.distributed as dist
    from ecg_denoise_b200 import _lib, synth
    from ecg_denoise_b200.engine import FusedTrainer

    world, rank, local_rank, dev = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch

    model, sd = bench_state_dict()
    model = model.to(dev)
    NB = 4                                       # rotating input batches (different windows every step)
    noisy, clean = synth.make_batch(NB * B, 2, 256, seed=2023 + 17 * rank)
    hx = torch.from_numpy(noisy).view(NB, B, 2, 256).pin_memory()
    ht = torch.from_numpy(clean).view(NB, B, 2, 256).pin_memory()
    dx, dt = hx.to(dev), ht.to(dev)

    trainer = FusedTrainer(model, lr=1e-3, use_graph=(args.graph == "on"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- launches per step (counted once, un-graphed) ---------------------------------------------------
    eager = FusedTrainer(model, lr=1e-3, use_graph=False)
    eager.step(dx[0], dt[0])
    torch.cuda.synchronize()
    _lib.launch_count(reset=True)
    eager.step(dx[1], dt[1])
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count(reset=True)

    # ---- device-resident timing -------------------------------------------------------------------------
    for i in range(args.warmup):
        trainer.step(dx[i % NB], dt[i % NB])
    barrier()
    stop = threading.Event()
    clk_path = os.path.join(tempfile.gettempdir(), f"clocks_{os.getpid()}.csv")
    th = threading.Thread(target=sample_clocks, args=(stop, clk_path), daemon=True)
    if rank == 0:
        th.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        loss, rmse, snr, out = trainer.step(dx[i % NB], dt[i % NB])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    final_loss = float(loss.item())
    if args.dump_outputs and rank == 0:           # before the end-to-end loop below trains the model further
        dump_outputs(args.dump_outputs, loss, rmse, snr, out, model)

    # ---- end to end: pinned host batch -> H2D -> step -> D2H loss ---------------------------------------
    for i in range(3):                            # warm-up of the same loop (staging buffers, copy stream, pinned slots)
        trainer.prefetch_host(hx[i % NB], ht[i % NB])
        trainer.read_async(trainer.step_host(hx[i % NB], ht[i % NB]))()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e2.record()
    # Software-pipelined loop: the copy of batch i + 1 runs on a copy stream under step i (the one-batch-ahead prefetch
    # of any pinned-memory input pipeline), and the loss of step i is read on the host after step i + 2 has been
    # enqueued, so the GPU does not idle on the host round trip.  Every step's inputs are copied from the host and every
    # step's loss is read by the host inside the timed region.
    # (two steps of slack: with one, a single host hiccup -- e.g. the driver lock taken by the nvidia-smi clock sampler
    #  above -- longer than a 2 ms step leaves the GPU idle; measured 50 us/step at 30 steps, tools/exp_e2e_gap.py)
    LAG = 2
    trainer.prefetch_host(hx[0], ht[0])
    pending = []
    for i in range(args.steps):
        l = trainer.step_host(hx[i % NB], ht[i % NB])
        pending.append(trainer.read_async(l))     # device -> host read of this step's result, collected LAG steps later
        trainer.prefetch_host(hx[(i + 1) % NB], ht[(i + 1) % NB])
        if len(pending) > LAG:
            host_loss = pending.pop(0)()
    while pending:
        host_loss = pending.pop(0)()
    e3.record()
    barrier()
    ms_e2e = max(e2.elapsed_time(e3), 1e3 * (time.perf_counter() - t0))
    if rank == 0:
        time.sleep(0.2)
        stop.set()
        th.join(timeout=10)

    ms, ms_e2e = max_over_ranks([ms, ms_e2e], dev, world)
    peaks = load_peaks()
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_hbm = peaks.get("hbm_gbs", 6500.0)
    peak_src = ("measured (MEASURED_PEAKS.json: bf16_tflops_sustained, hbm_gbs)" if peaks
                else "fallback (B200_PROFILING.md): 1.4 PFLOP/s sustained bf16, 6.5 TB/s HBM copy")

    # ---- per-kernel timing (roofline pass; un-graphed, events after every launch) ------------------------
    # (under torch.distributed every rank runs it -- the eager step contains the collectives -- and rank 0 reports)
    roofline, table = None, None
    if not args.no_profile:
        lib = _lib.load()
        st = torch.cuda.current_stream().cuda_stream
        agg = {}
        reps = 3
        for r in range(reps):
            torch.cuda.synchronize()
            _lib.check(lib.ralenet_profile_begin(ctypes.c_void_p(st)))
            eager.step(dx[r % NB], dt[r % NB])
            n_max = 8192
            labels = ctypes.create_string_buffer(n_max * 48)
            msb = (ctypes.c_float * n_max)()
            n = lib.ralenet_profile_end(labels, 48, msb, n_max)
            for i in range(n):
                lab = labels.raw[i * 48:(i + 1) * 48].split(b"\0")[0].decode()
                a = agg.setdefault(lab, [0, 0.0])
                a[0] += 1
                a[1] += msb[i]
        total = sum(a[1] for a in agg.values())
        table = sorted(((lab, a[0] // reps, a[1] / a[0], a[1] / reps) for lab, a in agg.items()), key=lambda r: -r[3])
        top, flops, nbytes = None, None, None
        for row in table:                      # dominant kernel with matmul-shaped algorithmic work
            f, nb = algorithmic_work(row[0], B)
            if f:
                top, flops, nbytes = row, f, nb
                break
        if top is not None:
            traffic, traffic_src = None, None
            try:     # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
                tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
                e = tr.get(top[0])
                if e and B == PER_GPU_BATCH:
                    traffic, traffic_src = e["dram_bytes_per_launch"], "profiles/" + os.path.basename(e["source"])
            except (OSError, ValueError, KeyError):
                pass
            secs = top[2] * 1e-3
            ach_tf, ach_gb = flops / secs / 1e12, nbytes / secs / 1e9
            # which roof binds: the kernel's FLOP per byte (measured DRAM traffic if captured, else algorithmic
            # bytes) against the ridge of the measured peaks
            intensity = flops / (traffic if traffic else nbytes)
            ridge = peak_tf * 1e12 / (peak_hbm * 1e9)
            hbm_bound = intensity < ridge
            roofline = {"kernel": top[0], "bound": "hbm" if hbm_bound else "tensor",
                        "achieved": ach_gb if hbm_bound else ach_tf, "peak": peak_hbm if hbm_bound else peak_tf,
                        "unit": "GB/s" if hbm_bound else "TFLOP/s",
                        "frac": (ach_gb / peak_hbm) if hbm_bound else (ach_tf / peak_tf),
                        "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": nbytes, "algorithmic_flops_per_launch": flops,
                        "flop_per_byte": intensity, "ridge_flop_per_byte": ridge,
                        "tensor_view": {"achieved_tflops": ach_tf, "peak_tflops": peak_tf, "frac": ach_tf / peak_tf},
                        "hbm_view": {"achieved_GBs": ach_gb, "peak_GBs": peak_hbm, "frac": ach_gb / peak_hbm},
                        "avg_launch_ms": top[2], "launches_per_step": top[1], "share_of_step": top[3] / (total / reps),
                        "note": "algorithmic bytes = fp32 block input/output + the tensors saved for the backward; "
                                "algorithmic FLOPs = 2*MAC of the projections and of q.k^T / p.v (and adjoints); both "
                                "over the live per-launch time of the un-graphed step (CUDA events on the launch "
                                "stream).  The bound is chosen by the kernel's FLOP/byte against the ridge; the kernel "
                                "is in fact issue-/latency-bound well below both roofs (DESIGN.md section 4)"}
        if args.dump_kernels and rank == 0:
            with open(args.dump_kernels, "w") as f:
                json.dump({"per_step_ms_sum": total / reps, "kernels": [
                    {"label": l, "launches_per_step": c, "avg_ms": a, "ms_per_step": s} for l, c, a, s in table]}, f,
                    indent=1)

    comm_kind = None
    if world > 1:
        c = getattr(model._plan, "_comm", None)
        comm_kind = c.kind if c is not None else "NCCL all-reduce (torch.distributed) captured in the step graph"
    value = world * B * args.steps / (ms * 1e-3)
    per_gpu = value / world
    whole = {"flops_per_window": FLOPS_PER_WINDOW_TRAIN, "bytes_per_window": BYTES_PER_WINDOW_TRAIN,
             "tflops_per_gpu": per_gpu * FLOPS_PER_WINDOW_TRAIN / 1e12,
             "frac_of_bf16_sustained": per_gpu * FLOPS_PER_WINDOW_TRAIN / 1e12 / peak_tf,
             "hbm_GBs_per_gpu": (per_gpu * BYTES_PER_WINDOW_TRAIN + ADAM_BYTES_PER_STEP * 1e3 / (ms / args.steps)) / 1e9,
             "frac_of_hbm": (per_gpu * BYTES_PER_WINDOW_TRAIN + ADAM_BYTES_PER_STEP * 1e3 / (ms / args.steps)) / 1e9 / peak_hbm,
             "note": "algorithmic FLOPs (reference flop count) and fp32-activation HBM bytes of SURVEY 8d over the "
                     "measured step; the fp32 roofline of that schedule is 2.79 M windows/s per GPU"}

    # ---- sub-records: the north star's other configs, same run ----------------------------------------------
    extras = {}
    trainer.close()
    eager.close()
    del trainer, eager

    def guarded(name, fn):
        try:
            extras[name] = fn()
        except Exception as e:      # noqa: BLE001 -- a failing sub-record must not lose the headline line
            if world > 1:
                raise                # ranks must stay in lock step; fail loudly under torchrun
            extras[name] = {"error": f"{type(e).__name__}: {e}"[:300]}

    if not args.no_extras:
        sub_steps = max(5, min(args.steps, 10))
        guarded("config4", lambda: config4_record(dev, sd, world, rank, sub_steps, 3, barrier))
        if world > 1:
            guarded("dp_parity", lambda: dp_parity_record(dev, sd, world, rank))
        guarded("inference", lambda: inference_record(model, dev, world, rank, 3, 2))
        if world == 1:
            guarded("config3", lambda: train12_record(dev, world, rank, sub_steps, 3))
            guarded("dropin", lambda: dropin_record(dev, sd, B, sub_steps, 3))
            guarded("eager_gpu_baseline", lambda: eager_gpu_baseline(dev, sd, B))

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = time_cpu_baseline()

    if rank == 0:
        clocks = parse_clocks(clk_path, local_rank)
        bytes_in = 2 * B * 2 * 256 * 4
        cfg = workload_config(world, B)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "e2e": {"value": world * B * args.steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": bytes_in,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                    "loop": "FusedTrainer.step_host from pinned host batches; batch i+1 copied on a copy stream under "
                            "step i (prefetch_host), the loss of step i read on the host after step i+2 is enqueued "
                            "(read_async); every copy and every read inside the timed region"},
            "gpu_launches": launches_per_step * args.steps, "launches_per_step": launches_per_step,
            "clocks": clocks, "final_loss": final_loss, "cuda_graph": args.graph == "on", "exchange": comm_kind,
            "roofline": roofline, "whole_step": whole, "cpu_baseline": cpu_base,
        }
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
