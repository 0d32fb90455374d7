#!/usr/bin/env python
"""Times the inverse flow against the forward on 2^22 points, for cfg2 (8-D PWLin) and the configs[3] flow (8-D PWQuad),
in both BatchNorm modes: CUDA events around whole calls (after warm-up), and the per-launch device times of one call
from the library's timing sink (nis_flow_timing_begin / _end), grouped by launch tag.  Columns: forward, inverse on the
fp16-split tensor-core kernel, inverse on the shape-generic kernel (NIS_TC=0, fewer repetitions).  Prints the GPU's name
and power limit first.  Usage: time_inverse.py [log2 points]"""
import ctypes
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from nf_b200 import _cabi  # noqa: E402
from nf_b200.normalizing_flows.manager import PWLinManager, PWQuadManager  # noqa: E402

TAGS = {0: "pack", 1: "column moments", 2: "other", 10: "fused cell", 11: "layer pass (state)", 12: "final pass (stored)",
        13: "layer pass (stored)"}


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def per_launch(fn):
    lib = _cabi.lib()
    lib.nis_flow_timing_begin(_cabi.stream_ptr())
    fn()
    ms = (ctypes.c_float * 512)()
    tags = (ctypes.c_int32 * 512)()
    n = lib.nis_flow_timing_end(ms, tags, 512)
    per = {}
    for i in range(max(n, 0)):
        per.setdefault(int(tags[i]), []).append(float(ms[i]))
    return ", ".join("%s %d x %.3f ms" % (TAGS.get(t, str(t)), len(v), sum(v) / len(v)) for t, v in sorted(per.items()))


def main():
    n = 1 << (int(sys.argv[1]) if len(sys.argv) > 1 else 22)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print("GPU: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), smi[0] if smi else "n/a"))
    print("points: %d" % n)
    for kind in ("lin", "quad"):
        torch.manual_seed(1234)
        if kind == "lin":
            NF = PWLinManager(n_flow=8)
            NF.create_model(4, 6, 32, [64] * 3, 4)
            name = "cfg2 (PWLin)"
        else:
            NF = PWQuadManager(n_flow=8)
            NF.create_model(6, 32, [64] * 3)
            name = "cfg4 (PWQuad)"
        x = torch.rand(n, 8, device="cuda", dtype=torch.float32)
        for mode in ("eval", "train"):
            model = NF._model.train(mode == "train")
            spec = model.spec()
            train = mode == "train"
            with torch.no_grad():
                y = model(x).detach()
                fwd = timed(lambda: model(x), 3, 10)
                fwd_l = per_launch(lambda: model(x))
                inv = timed(lambda: spec.inverse(y, train), 3, 10)
                inv_l = per_launch(lambda: spec.inverse(y, train))
                os.environ["NIS_TC"] = "0"
                try:
                    gen = timed(lambda: spec.inverse(y, train), 1, 2)
                finally:
                    del os.environ["NIS_TC"]
            print("%s %s: forward %.3f ms | tensor-core inverse %.3f ms (%.2fx forward) | generic inverse %.3f ms" % (
                name, mode, fwd, inv, inv / fwd, gen))
            print("    forward launches: " + fwd_l)
            print("    inverse launches: " + inv_l)


if __name__ == "__main__":
    main()
