#!/usr/bin/env python
"""Times the cfg2 flow forward (eval and train BN) on 2^22 points with CUDA events; honours the tuning
environment knobs of the library (NIS_TC, NIS_DISABLE_TILED).  Development aid."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from nf_b200.normalizing_flows.manager import PWLinManager, PWQuadManager  # noqa: E402

n = 1 << (int(sys.argv[1]) if len(sys.argv) > 1 else 22)
torch.manual_seed(1234)
kind = sys.argv[2] if len(sys.argv) > 2 else "lin"
if kind == "lin":
    NF = PWLinManager(n_flow=8)
    NF.create_model(4, 6, 32, [64] * 3, 4)
else:
    NF = PWQuadManager(n_flow=8)
    NF.create_model(6, 32, [64] * 3)
x = torch.rand(n, 8, device="cuda", dtype=torch.float32)
for mode in ("eval", "train"):
    model = NF._model.train(mode == "train")
    with torch.no_grad():
        for _ in range(3):
            model(x)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            model(x)
        e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    print(kind + " NIS_TC=%s NIS_DISABLE_TILED=%s mode=%s: %.3f ms  %.3e pts/s  %.1f TFLOP/s algorithmic" % (
        os.environ.get("NIS_TC", "1"), os.environ.get("NIS_DISABLE_TILED", "0"), mode, ms, n / ms * 1e3,
        n * 199680 / ms / 1e9))
