#!/usr/bin/env python
"""Benchmark of the NIS hot path (BASELINE.json): fused flow forward + log-det, points/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (N=1 and per GPU for N>1, weak scaling): BASELINE.json configs[1] — 8D, PWLinear coupling,
6 cells, 32 bins, conditioner [64]*3, forward + Jacobian on 2^22 synthetic uniform points per step,
BatchNorm in train mode (batch statistics) exactly as the reference's integrate() runs it
(manager.py:397).  A step = one pass of the flow over the 2^22-point batch (+ for N>1 the moment
reduction and its NCCL all-reduce, the path's only exchange).  One JSON line is printed by rank 0.

Extra objects on the line: ``roofline`` (dominant kernel vs the measured FP32-FMA peak — this path is
compute-bound on the FP32 pipe, SURVEY.md §8d — plus its HBM view), ``cpu_baseline`` (the oracle port of
the reference timed on the host cores on a bounded sample), ``e2e`` (same metric through the public API
from pinned host buffers, H2D/D2H inside the timed region), ``eval_mode`` (BN folded: one launch),
``rambo`` (BASELINE.json configs[2]: events/s of the fused RAMBO+cuts kernel against the HBM roofline).
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

CFG2 = dict(kind="lin", n_flow=8, n_pass_through=4, n_cells=6, n_bins=32, NN=[64] * 3, roll_step=4)
N_POINTS = 1 << 22
FLOP_PER_POINT = 199680          # SURVEY.md §8(d): 6 cells x 2 x 16 640 MAC
IO_BYTES_PER_POINT = 68          # fp32 in 32 B + out 36 B
RAMBO_EVENTS = 1 << 24
RAMBO_BYTES_PER_EVENT = 264      # fp64: 8 uniforms in + (6x4 momenta + weight) out
METRIC = "nis_flow_fwd_logdet_points_per_sec"
DUMP_ROWS = 1 << 20              # --dump-outputs: 2^20 of the 2^22 output rows, 36 MB of float32
DUMP_SEED = 2027


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_flow(seed=1234):
    from nf_b200.normalizing_flows.manager import PWLinManager
    torch.manual_seed(seed)
    NF = PWLinManager(n_flow=CFG2["n_flow"])
    NF.create_model(CFG2["n_pass_through"], CFG2["n_cells"], CFG2["n_bins"], CFG2["NN"], CFG2["roll_step"])
    if torch.cuda.is_available():
        NF._model.to(torch.device("cuda", torch.cuda.current_device()))     # this rank's GPU (create_model uses cuda:0)
    return NF


def time_steps(fn, steps, warmup, world, join=None):
    """W untimed + exactly K timed steps, barrier + synchronize on both sides, CUDA events, max over ranks.
    ``join`` (optional) makes the timing stream wait for side streams before the end event is recorded."""
    for _ in range(warmup):
        fn()
    if join:
        join()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    if join:
        join()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / steps


def dump_outputs(path, XJ):
    """Writes what one flow step returns to its caller, XJ [N, 9] (the eight mapped coordinates, then the Jacobian),
    as path/xj.npy (float32), so that two builds can be compared output for output.  The whole output is larger than
    a comparison needs, so the rows written are a fixed sample: DUMP_ROWS distinct row indices drawn with DUMP_SEED,
    in increasing order."""
    rows = torch.randperm(XJ.shape[0], generator=torch.Generator().manual_seed(DUMP_SEED))[:DUMP_ROWS].sort().values
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "xj.npy"), XJ.index_select(0, rows.to(XJ.device)).float().cpu().numpy())


def fma_peak_tflops():
    from nf_b200 import _cabi
    lib = _cabi.lib()
    out = torch.zeros(4, device="cuda")
    best = 0.0
    for it in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        flop = lib.nis_probe_fp32_fma(_cabi.ptr(out), 1 << 15, _cabi.stream_ptr())
        e1.record()
        torch.cuda.synchronize()
        if it:
            best = max(best, flop / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def tensor_peak_tflops(kind, n):
    """Measured tcgen05.mma peak (TFLOP/s, all SMs) for kind 0 = kind::tf32 / 1 = kind::f16 at M = 128, N = n, A in
    tensor memory: nis_probe_tensor issues 8192 back-to-back MMAs per SM; best of 5 after one warm-up."""
    from nf_b200 import _cabi
    lib = _cabi.lib()
    best = 0.0
    for it in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        flop = lib.nis_probe_tensor(kind, n, 1024, _cabi.stream_ptr())
        e1.record()
        torch.cuda.synchronize()
        if flop <= 0:
            return None
        if it:
            best = max(best, flop / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def pcie_probe(dev, nbytes=1 << 28):
    """Host<->device copy bandwidth of this box from pinned memory (GB/s): H2D alone, D2H alone, and both at once on
    two streams - the ceiling of the end-to-end number, which moves 285 MB per step across PCIe."""
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def timed(do_in, do_out):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            if do_in:
                with torch.cuda.stream(s1):
                    d_in.copy_(h_in, non_blocking=True)
            if do_out:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize()
        return 3 * nbytes * (int(do_in) + int(do_out)) / (time.perf_counter() - t0) / 1e9

    timed(True, True)
    return {"h2d_gbs": timed(True, False), "d2h_gbs": timed(False, True), "both_directions_total_gbs": timed(True, True)}


LAUNCH_NAMES = {0: "weight packs", 1: "flow_col_moments_kernel", 11: "flow_cell_h_kernel<.,.,1> layer pass from the state",
                13: "flow_cell_h_kernel<.,.,3> layer pass from stored activations",
                12: "flow_cell_h_kernel<.,.,2> final pass (output layer + splines)", 10: "flow_cell_h_kernel<.,.,0> fused cell",
                2: "other"}


def count_flow_launches(model, x, dev):
    """Kernels the library launches for one forward (its own event marks, nis_flow_timing_begin / _end)."""
    import ctypes
    from nf_b200 import _cabi
    lib = _cabi.lib()
    lib.nis_flow_timing_begin(_cabi.stream_ptr(dev))
    with torch.no_grad():
        model(x)
    lms = (ctypes.c_float * 512)()
    ltag = (ctypes.c_int32 * 512)()
    return max(int(lib.nis_flow_timing_end(lms, ltag, 512)), 0)


def flow_launch_times(model, x, dev, n_points, hbm_peak, abytes, traffic=None):
    """Per-launch device times of ONE forward, from CUDA events the library records on the launch stream around every
    kernel (nis_flow_timing_begin / _end), grouped by kernel: launches, average ms, share of the step and - with the
    algorithmic bytes per point of each launch - the achieved GB/s against the measured HBM peak."""
    import ctypes
    from nf_b200 import _cabi
    lib = _cabi.lib()
    lib.nis_flow_timing_begin(_cabi.stream_ptr(dev))
    with torch.no_grad():
        model(x)
    lms = (ctypes.c_float * 512)()
    ltag = (ctypes.c_int32 * 512)()
    nl = lib.nis_flow_timing_end(lms, ltag, 512)
    per = {}
    for i in range(max(nl, 0)):
        per.setdefault(int(ltag[i]), []).append(float(lms[i]))
    tot_ms = sum(sum(v) for v in per.values()) or 1.0
    kernels = []
    for tag, v in sorted(per.items(), key=lambda kv: -sum(kv[1])):
        k = {"kernel": LAUNCH_NAMES.get(tag, str(tag)), "launches_per_step": len(v), "avg_ms": sum(v) / len(v),
             "share_of_step": sum(v) / tot_ms}
        if tag in abytes:
            g = n_points * abytes[tag] / (k["avg_ms"] * 1e-3) / 1e9
            k.update({"algorithmic_bytes_per_point": abytes[tag], "achieved_gbs": g, "frac_of_hbm_peak": g / hbm_peak,
                      "traffic": (traffic or {}).get(tag)})
        kernels.append(k)
    return kernels


def parity_checks(rank, world, dev):
    """Run by every `bench.py --gpus N` (VERDICT r1 item 2): the N-rank paths checked in the driver's own run.
    (a) data-parallel gradient == single-GPU gradient: every rank backpropagates the variance loss of ITS minibatch
        (per-rank BN statistics), the flat gradient is sum-allreduced; rank 0 also computes all `world` minibatches
        one after the other on its own GPU and sums — the two must agree (SURVEY 8e);
    (b) per-rank latent streams differ under identical seeding;
    (c) the configs[3] integrate result is finite and within one honest standard error (filled in by main)."""
    from nf_b200.normalizing_flows.manager import BasicManager, PWLinManager
    torch.manual_seed(77)
    NF = PWLinManager(n_flow=8)
    NF.create_model(4, 3, 32, [64, 64], 4)
    NF._model.to(dev)
    model = NF._model.train()
    params = list(model.parameters())

    def minibatch(r):
        g = torch.Generator().manual_seed(4242 + r)
        return torch.rand(4096, 8, generator=g, dtype=torch.float32).to(dev)

    def grad_of(x):
        model.zero_grad()
        XJ = model(x)
        f = torch.exp(-((XJ[:, :-1].detach() - 0.5) ** 2).sum(-1) / 0.3)
        (torch.var(f * XJ[:, -1]) / world).backward()
        return torch.cat([p.grad.reshape(-1) for p in params]).clone()

    out = {}
    mine = grad_of(minibatch(rank))
    if world > 1:
        BasicManager._allreduce_grads(params)
        reduced = torch.cat([p.grad.reshape(-1) for p in params]).clone()
    else:
        reduced = mine
    if rank == 0:
        ref = sum(grad_of(minibatch(r)) for r in range(world))
        out["dp_gradient_max_err_over_scale"] = float((reduced - ref).abs().max() / ref.abs().max())
        out["dp_gradient_ok"] = out["dp_gradient_max_err_over_scale"] <= 2e-4
    torch.manual_seed(99)
    gen = BasicManager._rank_generator(dev, rank, world)
    pts = torch.rand(8, device=dev, generator=gen)
    if world > 1:
        allp = [torch.zeros_like(pts) for _ in range(world)]
        dist.all_gather(allp, pts)
        out["rank_streams_differ"] = all(not torch.equal(allp[0], a) for a in allp[1:])
    return out


def reference_flow(threads):
    """The reference's CPU path for this workload as a callable [B,9] float64 -> [B,9] (train-mode BN like
    the reference's integrate).  kind "reference": the UNMODIFIED reference package installed under
    baseline/_ref (pip --target from /root/reference; git-ignored, travels with the repo snapshot), built
    through its own PWLinManager.create_model (plus the documented .double() shim, SURVEY.md §8c).
    kind "port": the oracle restatement, used when baseline/_ref is absent."""
    torch.set_num_threads(threads)
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "nisrep")):
        sys.path.insert(0, ref)
        try:
            from nisrep.normalizing_flows.manager import PWLinManager as RefPWLin
            torch.manual_seed(1234)
            NF = RefPWLin(n_flow=CFG2["n_flow"])
            try:
                NF.create_model(CFG2["n_pass_through"], CFG2["n_cells"], CFG2["n_bins"], CFG2["NN"], CFG2["roll_step"])
            except RuntimeError:
                pass                     # mixed-dtype trial forward, raised after _model is built (manager.py:493-499)
            model = NF._model.to("cpu").double()
            model.train()
            return (lambda xj: model(xj)), "reference"
        except Exception as e:           # fall through to the port, but say why
            print("reference import failed, using the oracle port: %r" % (e,), file=sys.stderr)
    from oracle import flow as oflow
    layers = oflow.pwlin_layers(CFG2["n_flow"], CFG2["n_pass_through"], CFG2["n_cells"], CFG2["roll_step"])
    cells, _ = oflow.compile_layers(layers, CFG2["n_flow"])
    sd = oflow.init_state_dict(cells, CFG2["n_flow"], "lin", CFG2["n_bins"], CFG2["NN"], seed=1234)
    return (lambda xj: oflow.flow_forward(layers, sd, xj, "lin", CFG2["n_bins"], train=True)[0]), "port"


def cpu_reference_flow(n_points, reps, threads):
    fn, kind = reference_flow(threads)
    x = torch.rand(n_points, CFG2["n_flow"], dtype=torch.float64)
    xj = torch.cat((x, torch.ones(n_points, 1, dtype=torch.float64)), 1)
    best = None
    with torch.no_grad():
        for i in range(reps + 1):
            t0 = time.perf_counter()
            fn(xj)
            dt = time.perf_counter() - t0
            if i and (best is None or dt < best):
                best = dt
    return n_points / best, best, kind


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores, same
    metric/config; each step is a bounded sample of the workload.  Rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    sample = 1 << 19                     # ~2.4 s per step on 16 host threads: a 10+3-step run stays near half a minute
    fn, kind = reference_flow(threads)
    x = torch.rand(sample, CFG2["n_flow"], dtype=torch.float64)
    xj = torch.cat((x, torch.ones(sample, 1, dtype=torch.float64)), 1)
    with torch.no_grad():
        for _ in range(args.warmup):
            fn(xj)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn(xj)
        dt = (time.perf_counter() - t0) / args.steps
    value = sample / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(sample),
            "cpu_baseline": {"value": value, "unit": "points/s", "cores": threads, "kind": kind,
                             "sample": "%d points per step (of the 2^22-point workload), float64, train-mode BN" % sample},
            "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(points):
    return {"workload": "cfg2: 8D PWLinear flow, 6 cells, 32 bins, MLP [64]*3, forward + log-det, "
                        "train-mode BatchNorm (batch statistics, as the reference's integrate runs it)",
            "points_per_step_per_gpu": points, "n_flow": 8, "cells": 6, "bins": 32, "hidden": [64, 64, 64],
            "l2": "inputs larger than L2 (134 MB fp32 points per step > 126 MB)"}


def bench_train_step(steps, warmup, world, dev, log2n=16):
    """SURVEY.md 8(d)(iii): variance-loss training step of the cfg2 flow — forward + backward (tcgen05 kernels
    of flow_tc.cu / flow_bwd_tc.cu) on a per-rank minibatch of 2^log2n points, gradient sum-allreduce (NCCL)
    when N > 1."""
    from nf_b200.normalizing_flows.manager import BasicManager
    NF = build_flow()
    model = NF._model.train()
    params = list(model.parameters())
    n = 1 << log2n
    x = torch.rand(n, 8, device=dev, dtype=torch.float32)
    f = torch.exp(-((x - 0.5) ** 2).sum(-1) / 0.2)

    def step():
        model.zero_grad()                 # set_to_none, as the training loop does (manager.py): gradients land as views of one flat buffer
        XJ = model(x)
        torch.var(f * XJ[:, -1]).backward()
        if world > 1:
            BasicManager._allreduce_grads(params)

    ms = time_steps(step, steps, warmup, world)
    return {"metric": "nis_train_step_points_per_sec", "value": world * n / (ms * 1e-3), "unit": "points/s",
            "ms_per_step": ms, "config": {"workload": "cfg2 flow, variance loss, forward + backward on the tcgen05 "
                                          "kernels (+ gradient all-reduce), 2^%d points per rank per step" % log2n}}


def bench_readme(dev):
    """BASELINE configs[0], the reference's README example: 2-D camel, PWQuadManager, 4 bins, MLP [3]*3, 10000
    points per batch, 300 epochs of Adamax variance training through _train_variance_forward_seq, then integrate.
    Latency-bound (shape-generic kernels, ~50 launches per epoch); wall seconds on rank 0."""
    import tempfile
    from nf_b200.normalizing_flows.manager import PWQuadManager

    def camel(x):
        return torch.exp(-((x[:, 0] - 0.75) ** 2 + (x[:, 1] - 0.75) ** 2) / (0.2 ** 2)) + \
            torch.exp(-((x[:, 0] - 0.25) ** 2 + (x[:, 1] - 0.25) ** 2) / (0.2 ** 2))

    # four runs: the first run of a process also pays for loading the kernels and the optimizer's / integrand's torch kernels
    # it is the first to use (CUDA loads modules lazily) - reported as first_run_seconds; `value` is the median of the
    # three warm runs (the example is host-latency sensitive - 300 epochs of ~1 ms with a loss read-back each - and single
    # runs on a shared VM scatter by a factor of two; all four are listed in runs_seconds)
    gc.collect()
    torch.cuda.empty_cache()                  # cached blocks of the previous (GB-sized) workloads
    runs = []
    for _ in range(4):
        torch.manual_seed(0)
        NF = PWQuadManager(n_flow=2)
        NF.create_model(2, 4, [3] * 3, dev=dev.index or 0)
        optim = torch.optim.Adamax(NF._model.parameters(), lr=2e-3, weight_decay=1e-04)
        torch.cuda.synchronize()
        t0 = time.time()
        NF._train_variance_forward_seq(camel, optim, True, tempfile.mkdtemp(), 10000, 300, dev.index or 0, False, True, preburn_time=50)
        torch.cuda.synchronize()
        t1 = time.time()
        sig, err = NF.integrate(camel, 10, 10000, dev.index or 0)
        torch.cuda.synchronize()
        runs.append((t1 - t0, time.time() - t1, float(sig), float(err), float(NF.best_loss), float(NF.int_loss)))
        del NF, optim
    warm = sorted(runs[1:], key=lambda r: r[0])
    w = warm[len(warm) // 2]
    return {"metric": "readme_example_wall_seconds", "value": w[0], "unit": "s", "higher_is_better": False,
            "first_run_seconds": runs[0][0], "runs_seconds": [r[0] for r in runs],
            "us_per_minibatch_step": w[0] / (300 * 5) * 1e6,
            "integrate_seconds": w[1], "estimate": w[2], "reported_error": w[3],
            "analytic": 0.232322, "best_loss": w[4], "int_loss": w[5],
            "same_result_every_run": all(r[2:] == runs[0][2:] for r in runs),
            "reference": "368 s on 8 CPU cores, best_loss 0.024 from int_loss 0.071 (BASELINE.md)"}


def bench_wide(steps, warmup, world, dev):
    """BASELINE configs[4]: 16-D PWQuad flow, 8 mask cells, 64 bins, MLP [256]*4 (the tensor-core conditioner path:
    flow_wide.cu / flow_bwd_wide.cu) — forward + log-det with train-mode BN, and one variance-loss training step
    (forward + backward + gradient all-reduce), 2^16 points per rank per step."""
    from nf_b200 import _cabi
    from nf_b200.normalizing_flows.manager import BasicManager, PWQuadManager
    torch.manual_seed(1234)
    NF = PWQuadManager(n_flow=16)
    NF.create_model(8, 64, [256] * 4, dev=dev.index or 0)
    model = NF._model.train()
    params = list(model.parameters())
    n = 1 << 16
    flop = 8 * 2 * 462848                                    # SURVEY.md 8(d): 7.41 MFLOP per point forward
    x = torch.rand(n, 16, device=dev, dtype=torch.float32)
    f = torch.exp(-((x - 0.5) ** 2).sum(-1) / 0.4)

    def fwd():
        with torch.no_grad():
            model(x)

    def step():
        model.zero_grad()
        XJ = model(x)
        torch.var(f * XJ[:, -1]).backward()
        if world > 1:
            BasicManager._allreduce_grads(params)

    ms_f = time_steps(fwd, steps, warmup, world)
    ms_s = time_steps(step, steps, warmup, world)
    tf32_peak = tensor_peak_tflops(0, 128) or peaks()[0].get("bf16_tflops", 1590.0) / 2     # measured kind::tf32 peak
    ach = world * n * flop * 3 / (ms_f * 1e-3) / 1e12         # executed TF32 flops (3xTF32 split)
    return {"metric": "nis_flow_fwd_logdet_points_per_sec", "value": world * n / (ms_f * 1e-3), "unit": "points/s",
            "ms_per_step": ms_f,
            "config": {"workload": "configs[4]: 16-D PWQuad flow, 8 cells, 64 bins, MLP [256]*4, train-mode BN, 2^16 points per rank"},
            "roofline": {"bound": "tensor", "achieved": ach / world, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / world / tf32_peak,
                         "algorithmic_tflops": ach / 3 / world,
                         "peak_kind": "tcgen05.mma kind::tf32 M128 N128 K8 back to back on every SM, measured in this run",
                         "note": "3xTF32: three tensor MACs per conditioner MAC"},
            "train_step": {"metric": "nis_train_step_points_per_sec", "value": world * n / (ms_s * 1e-3), "unit": "points/s",
                           "ms_per_step": ms_s,
                           "activation_cache_bytes_per_rank": 4 * model.spec().act_saved_count(_cabi.lib(), n)}}


def bench_integrate(world, dev):
    """SURVEY.md 8(d)(iv) / BASELINE configs[3]: end-to-end NIS integrate — 8D PWQuad flow (6 mask cells, 32
    bins, [64]*3) -> RAMBO 2->4 massless at E_cm = 1000 -> |M|^2 = 1, through the public API
    (PWQuadManager.integrate + FlatInvertiblePhasespace); the estimate has the known answer
    0.0664828... (flat weight / 2s), since the flow is a bijection of the unit cube."""
    from nf_b200.normalizing_flows.manager import PWQuadManager
    from nf_b200.PhaseSpace.flat_phase_space_generator import FlatInvertiblePhasespace
    torch.manual_seed(1234)
    NF = PWQuadManager(n_flow=8)
    NF.create_model(6, 32, [64] * 3, dev=dev.index)
    ps = FlatInvertiblePhasespace([0.0] * 2, [0.0] * 4)
    ps.check_nan = False

    def f(X):
        return ps.generateKinematics_batch(1000.0, X, momenta=False)[1]

    # configs[3]: neval = 2^26 sharded over 8 GPUs -> 2^23 points per rank per iteration (weak scaling below 8 ranks)
    nitn, neval = 4, (1 << 23) * world
    NF.integrate(f, 1, neval, dev.index)                      # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sig, err = NF.integrate(f, nitn, neval, dev.index)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    honest = float(err) * nitn ** 0.5                          # manager.py:403 under-reports by sqrt(nitn)
    known = 0.06648282151394422
    xq = torch.rand(1 << 22, 8, device=dev, dtype=torch.float32)
    flow_k = flow_launch_times(NF.best_model, xq, dev, 1 << 22, peaks()[0]["hbm_gbs"],
                               {1: 36, 11: 36 + 256, 13: 512, 12: 256 + 72, 10: 72},       # PWQuad keeps the z_3 store
                               {11: 1175477000, 13: 2294614000, 12: 1374712000})           # profiles/r02_ncu_h_quad.md
    del xq
    return {"metric": "nis_integrate_points_per_sec", "value": nitn * neval / dt, "unit": "points/s",
            "flow_kernels_at_2p22_points": flow_k,
            "estimate": float(sig), "reported_error": float(err), "honest_error": honest, "known_answer": known,
            "finite": bool(torch.isfinite(sig)), "within_one_honest_error": bool(abs(float(sig) - known) <= honest),
            "n_nonfinite_weights": NF.n_nonfinite,
            "config": {"workload": "configs[3]: 8D PWQuad flow -> RAMBO 2->4 massless -> |M|^2=1, nitn=%d x neval=%d "
                                   "(2^23 per rank; 2^26 at 8 ranks) sharded over the ranks, sum-allreduce of the moments"
                                   % (nitn, neval)}}


def bench_rambo(steps, warmup, world, hbm_peak, peak_kind):
    from nf_b200.PhaseSpace.flat_phase_space_generator import FlatInvertiblePhasespace
    ps = FlatInvertiblePhasespace([100.0] * 2, [100.0] * 4, pdf=None, pdf_active=False)
    ps.check_nan = False
    r = torch.rand(RAMBO_EVENTS, 8, device="cuda", dtype=torch.float64)

    def step():
        ps.generateKinematics_batch(1000.0, r, pT_mincut=20, delR_mincut=0.4, rap_maxcut=2.5)

    ms = time_steps(step, steps, warmup, world)

    def step_w():
        ps.generateKinematics_batch(1000.0, r, pT_mincut=20, delR_mincut=0.4, rap_maxcut=2.5, momenta=False)

    ms_w = time_steps(step_w, steps, warmup, world)
    ev = world * RAMBO_EVENTS / (ms * 1e-3)
    gbs = RAMBO_EVENTS * RAMBO_BYTES_PER_EVENT / (ms * 1e-3) / 1e9
    del r
    return {"metric": "rambo_events_per_sec", "value": ev, "unit": "events/s", "ms_per_step": ms,
            "config": {"workload": "cfg3: FlatInvertiblePhasespace 2->4 massive (m=100), E_cm=1000, pdf inactive, "
                                   "pT>20, dR>0.4, |eta|<2.5 cuts", "events_per_step_per_gpu": RAMBO_EVENTS},
            "dtype": "f64",
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch at 2^24 events from the committed
                         # ncu --set full capture (profiles/r02_ncu_rambo.md: 1.074 GB + 3.304 GB); not re-measured per run
                         "traffic": 4376176000 if RAMBO_EVENTS == 1 << 24 else None,
                         "peak_kind": peak_kind, "algorithmic_bytes_per_event": RAMBO_BYTES_PER_EVENT},
            "weight_only": {"value": world * RAMBO_EVENTS / (ms_w * 1e-3), "unit": "events/s", "ms_per_step": ms_w}}


def bind_to_gpu_numa(local):
    """Host side of the end-to-end path: run this rank (and so first-touch its pinned staging buffers) on the CPUs of the
    NUMA node its GPU hangs off, as `numactl --cpunodebind` would.  With every rank on the default node the eight
    GPUs' copies share one socket's memory controllers.  Returns what it found (reported in the JSON line);
    BENCH_NUMA_BIND=0 turns it off."""
    info = {"numa_node": None, "cpus": None, "bound": False}
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        info["pci"] = bdf
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as fh:
            node = int(fh.read().strip())
        info["numa_node"] = node
        info["nodes_online"] = open("/sys/devices/system/node/online").read().strip()
        if node < 0 or os.environ.get("BENCH_NUMA_BIND", "1") == "0":
            return info
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info["cpus"] = len(cpus)
            info["bound"] = True
    except Exception as e:                                      # sysfs not there (container): leave the affinity alone
        info["error"] = repr(e)[:120]
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip cpu baseline / rambo / eval-mode extras")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of the rows the last step returned to DIR/xj.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local) if args.impl == "ours" else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL's banner / debug output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from nf_b200 import _cabi
    lib = _cabi.lib()
    pk, peak_kind = peaks()
    dev = torch.device("cuda", local)

    NF = build_flow()
    model = NF._model
    model.train()
    x = torch.rand(N_POINTS, 8, device=dev, dtype=torch.float32,
                   generator=torch.Generator(device=dev).manual_seed(2026 + rank))
    moments = torch.zeros(3, dtype=torch.double, device=dev)
    rws = torch.empty(lib.nis_reduce_workspace_bytes(), dtype=torch.uint8, device=dev)
    last = {}

    def step():
        with torch.no_grad():
            XJ = model(x)
        if world > 1:      # the path's only exchange: sum-allreduce of (sum J, sum J^2, n)
            J = XJ[:, -1].contiguous()
            lib.nis_reduce_moments(_cabi.ptr(J), _cabi.F32, J.numel(), _cabi.ptr(moments), 0, _cabi.ptr(rws),
                                   rws.numel(), _cabi.stream_ptr(dev))
            dist.all_reduce(moments)
        if args.dump_outputs:
            last["XJ"] = XJ
        return XJ

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = time_steps(step, args.steps, args.warmup, world)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["XJ"])
    last.clear()
    value = world * N_POINTS / (ms * 1e-3)
    n_cells, depth = 6, 3
    # counted, not assumed: the library marks every kernel it launches for one forward (two weight packs, the first cell's
    # column moments, per cell depth-1 layer passes and the final pass = 21 for cfg2) + the moments reduction at N > 1
    launches_per_step = count_flow_launches(model, x, dev) + (1 if world > 1 else 0)

    # ---- end to end through the public API from pinned host buffers ---------------------------------
    # Every step copies its 2^22 points host->device and its [2^22, 9] result device->host inside the timed
    # region.  The copies run on a side stream (double-buffered), so step i+1's upload and step i's download
    # overlap step i's / i+1's kernels; the timing stream joins both copy streams before the end event.
    xh = torch.rand(N_POINTS, 8, dtype=torch.float32).pin_memory()
    oh = torch.empty(N_POINTS, 9, dtype=torch.float32).pin_memory()
    xd = [torch.empty(N_POINTS, 8, device=dev, dtype=torch.float32) for _ in range(2)]
    h2d_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    ev_free = [torch.cuda.Event(), torch.cuda.Event()]      # input buffer i no longer read by the kernels
    ev_in = [torch.cuda.Event(), torch.cuda.Event()]        # input buffer i uploaded
    ev_out = torch.cuda.Event()
    state = {"i": 0, "keep": None, "k0": [], "k1": []}

    def step_e2e():
        i = state["i"] & 1
        first_use = state["i"] < 2
        state["i"] += 1
        main = torch.cuda.current_stream(dev)
        with torch.cuda.stream(h2d_stream):
            if not first_use:
                h2d_stream.wait_event(ev_free[i])
            xd[i].copy_(xh, non_blocking=True)
            ev_in[i].record(h2d_stream)
        main.wait_event(ev_in[i])
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(main)
        with torch.no_grad():
            out = model(xd[i])
        k1.record(main)
        state["k0"].append(k0)
        state["k1"].append(k1)
        ev_free[i].record(main)
        if world > 1:
            J = out[:, -1].contiguous()
            lib.nis_reduce_moments(_cabi.ptr(J), _cabi.F32, J.numel(), _cabi.ptr(moments), 0, _cabi.ptr(rws),
                                   rws.numel(), _cabi.stream_ptr(dev))
            dist.all_reduce(moments)
        ev_out.record(main)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(ev_out)
            oh.copy_(out, non_blocking=True)
        out.record_stream(d2h_stream)
        state["keep"] = out

    def join():
        main = torch.cuda.current_stream(dev)
        main.wait_stream(h2d_stream)
        main.wait_stream(d2h_stream)

    ms_e2e = time_steps(step_e2e, args.steps, args.warmup, world, join=join)
    kern_ms = [a.elapsed_time(b) for a, b in zip(state["k0"][-args.steps:], state["k1"][-args.steps:])]
    e2e = {"value": world * N_POINTS / (ms_e2e * 1e-3), "unit": "points/s", "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": xh.numel() * 4, "d2h_bytes_per_step": oh.numel() * 4,
           # the flow kernels alone, timed inside the end-to-end loop (while the copy engines move the neighbouring
           # steps' buffers): what the PCIe traffic costs the HBM-bound layer passes
           "kernels_ms_per_step_under_copies": sum(kern_ms) / max(len(kern_ms), 1),
           "api": "FlowSequential.__call__ (PWLinManager._model); pinned host float32 points in, pinned host "
                  "[N,9] result out, copies on a side stream inside the timed region"}
    del xh, oh, xd
    if world > 1:
        topo = [None] * world
        dist.all_gather_object(topo, numa)
    else:
        topo = [numa]
    e2e["host_topology"] = topo                                    # per rank: GPU PCI address, its NUMA node, CPUs bound to
    if rank == 0:
        e2e["pcie"] = pcie_probe(dev)
        e2e["pcie_bound_ms_per_step"] = (e2e["h2d_bytes_per_step"] + e2e["d2h_bytes_per_step"]) / \
            (e2e["pcie"]["both_directions_total_gbs"] * 1e9) * 1e3

    line = {"metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(N_POINTS),
            "e2e": e2e, "gpu_launches": launches_per_step * args.steps, "clocks": clocks}

    if rank == 0 or world > 1:
        fma = fma_peak_tflops()
        # dominant kernel: flow_cell_tc_kernel (tcgen05.mma kind::tf32, 3 products per conditioner MAC)
        tensor_flop_pt = n_cells * 3 * 2 * (64 * 64 * (depth - 1) + 64 * 128)      # executed on the tensor pipe
        tfl_exec = N_POINTS * tensor_flop_pt / (ms * 1e-3) / 1e12
        f16_peak = tensor_peak_tflops(1, 128) or pk["bf16_tflops"]
        f16_peak_n64 = tensor_peak_tflops(1, 64)
        tf32_meas = tensor_peak_tflops(0, 128)
        tfl = N_POINTS * FLOP_PER_POINT / (ms * 1e-3) / 1e12
        # moments pass reads the rows; first layer pass reads rows, writes z2; later passes read+write 256 B; final
        # first cell: column moments (36); every cell: layer pass from the state (36 + 256), depth-2 layer passes from stored
        # activations (the last one statistics only: no store), final pass (256 + 36 + 36, it also takes the next cell's moments)
        train_bytes_pt = 36 + n_cells * ((36 + 256) + (2 * (depth - 2) - 1) * 256 + (256 + 36 + 36))
        gbs_design = N_POINTS * train_bytes_pt / (ms * 1e-3) / 1e9
        gbs = N_POINTS * IO_BYTES_PER_POINT / (ms * 1e-3) / 1e9
        # ---- per-launch device times of one more forward (CUDA events recorded on the launch stream by the library:
        #      nis_flow_timing_begin / _end), outside the timed region -----------------------------------------------
        # algorithmic bytes per point of each launch: what the kernel has to read and write once (DESIGN.md 4.3)
        # (the last layer pass only takes statistics: it reads its 256 B/point tile and stores nothing)
        abytes = {1: 36, 11: 36 + 256, 13: 256, 12: 256 + 36 + 36, 10: 36 + 36}
        # dram__bytes_read.sum + dram__bytes_write.sum per launch at 2^22 points, ncu --set full (profiles/r02_ncu_h_kernel.md)
        traffic = {11: 1177050000, 13: 1239061000, 12: 1377346000, 10: 257961000} if N_POINTS == 1 << 22 else None
        kernels = flow_launch_times(model, x, dev, N_POINTS, pk["hbm_gbs"], abytes, traffic)
        dom = next((k for k in kernels if "achieved_gbs" in k), None)
        line["roofline"] = {
            # the dominant kernel of the train-mode step: an HBM-bound layer pass (reads one 256 B/point activation tile,
            # writes the next); achieved = algorithmic bytes of ONE launch / its device time measured in this run
            "bound": "hbm", "achieved": dom["achieved_gbs"] if dom else None, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": dom["frac_of_hbm_peak"] if dom else None, "traffic": dom.get("traffic") if dom else None,
            "peak_kind": "%s (MEASURED_PEAKS.json copy bandwidth)" % peak_kind,
            "kernel": dom["kernel"] if dom else None,
            "algorithmic_bytes_per_launch": N_POINTS * dom["algorithmic_bytes_per_point"] if dom else None,
            "kernels": kernels,
            "step": {
                "hbm_design": {"achieved": gbs_design, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs_design / pk["hbm_gbs"],
                               "bytes_per_point": train_bytes_pt,
                               "note": "all launches of the step: the train-mode layer-pass design moves the pre-BN activations "
                                       "through HBM once per BatchNorm layer (grid-wide statistics)"},
                "hbm_algorithmic": {"achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                                    "algorithmic_bytes_per_point": IO_BYTES_PER_POINT,
                                    "note": "SURVEY 8(d) I/O of the whole forward (32 B in + 36 B out)"},
                "tensor": {"achieved": tfl_exec, "peak": f16_peak, "unit": "TFLOP/s", "frac": tfl_exec / f16_peak,
                           "tensor_flop_per_point": tensor_flop_pt,
                           "peak_kind": "tcgen05.mma kind::f16 M128 N128 K16 back to back on every SM, measured in this run "
                                        "(nis_probe_tensor)",
                           "measured_tensor_peaks_tflops": {"f16_n128": f16_peak, "f16_n64": f16_peak_n64, "tf32_n128": tf32_meas,
                                                            "bf16_cublas_MEASURED_PEAKS": pk.get("bf16_tflops")},
                           "note": "executed fp16 flops (fp16-split operands: 3 tensor MACs per conditioner MAC); the step is "
                                   "not tensor-bound"},
                "fp32_equivalent": {"achieved": tfl, "peak": fma, "unit": "TFLOP/s", "frac": tfl / fma,
                                    "algorithmic_flop_per_point": FLOP_PER_POINT,
                                    "peak_kind": "FP32 FMA pipe measured in this run (nis_probe_fp32_fma): the roofline SURVEY 8(d) "
                                                 "states for this config; above 1 because the conditioner runs on the tensor pipe"}}}
        line["roofline"]["tensor_flop_per_point"] = tensor_flop_pt

    if not args.no_extras:
        model.eval()
        ms_eval = time_steps(step, args.steps, args.warmup, world)
        tfl_e = N_POINTS * FLOP_PER_POINT / (ms_eval * 1e-3) / 1e12
        tfl_e_exec = N_POINTS * line["roofline"]["tensor_flop_per_point"] / (ms_eval * 1e-3) / 1e12
        line["eval_mode"] = {"value": world * N_POINTS / (ms_eval * 1e-3), "unit": "points/s", "ms_per_step": ms_eval,
                             "launches_per_step": 2 + n_cells,
                             "roofline": {"bound": "tensor", "achieved": tfl_e_exec,
                                          "peak": line["roofline"]["step"]["tensor"]["peak"], "unit": "TFLOP/s",
                                          "frac": tfl_e_exec / line["roofline"]["step"]["tensor"]["peak"],
                                          "note": "fused eval cell: instruction-issue bound (profiles/r02_ncu_h_kernel.md), "
                                                  "neither tensor- nor HBM-bound",
                                          "fp32_equivalent": {"achieved": tfl_e, "peak": line["roofline"]["step"]["fp32_equivalent"]["peak"],
                                                              "frac": tfl_e / line["roofline"]["step"]["fp32_equivalent"]["peak"]}}}
        model.train()
        del x
        torch.cuda.empty_cache()
        line["rambo"] = bench_rambo(args.steps, args.warmup, world, pk["hbm_gbs"], peak_kind)
        line["train_step"] = bench_train_step(args.steps, args.warmup, world, dev)
        line["train_step_large"] = bench_train_step(args.steps, args.warmup, world, dev, log2n=20)
        line["integrate"] = bench_integrate(world, dev)
        par = parity_checks(rank, world, dev)
        par["integrate_finite"] = line["integrate"]["finite"]
        par["integrate_within_one_honest_error"] = line["integrate"]["within_one_honest_error"]
        line["parity"] = par
        line["wide_flow"] = bench_wide(args.steps, args.warmup, world, dev)
        if world == 1:
            line["readme_example"] = bench_readme(dev)
        if rank == 0 and world == 1:
            threads = os.cpu_count() or 1
            sample = 1 << 20                                # ~5 s per pass on 16 host threads: ~15 s of CPU work
            v, dt, kind = cpu_reference_flow(sample, 2, threads)
            line["cpu_baseline"] = {"value": v, "unit": "points/s", "cores": threads, "kind": kind,
                                    "sample": "%d points (of 2^22), best of 2 after 1 warm-up, float64, train-mode BN, "
                                              "torch CPU ops as the reference uses" % sample}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
