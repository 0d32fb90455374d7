"""Which kernel family runs each call: the kernels (names without template arguments) that one forward, the backward of
one forward + backward, and one inverse launch, recorded with torch.profiler, for shapes on each side of every choice the
host code makes (fp16-split / streamed-weights / register-tiled / shape-generic forward, cooperative small-batch kernels,
tensor-core / wide / shape-generic backward, the activation cache) and for the knobs that select the reference kernels."""
import re
from collections import Counter

import pytest
import torch

from gpu_util import make_manager

pytestmark = pytest.mark.gpu

CFG2 = dict(kind="lin", n_flow=8, n_pass_through=4, n_cells=6, n_bins=32, NN=[64] * 3, roll_step=4)
CFG4 = dict(kind="quad", n_flow=8, n_cells=6, n_bins=32, NN=[64] * 3)
CFG5_SMALL = dict(kind="quad", n_flow=16, n_cells=8, n_bins=16, NN=[128] * 2)
QUAD64_20BINS = dict(kind="quad", n_flow=8, n_cells=6, n_bins=20, NN=[64] * 3)
README = dict(kind="quad", n_flow=2, n_cells=2, n_bins=4, NN=[3] * 3)
AFFINE = dict(kind="affine", n_flow=8, n_pass_through=4, n_cells=4, n_bins=1, NN=[64] * 2, roll_step=4)
KNOBS = ("NIS_TC", "NIS_DISABLE_TILED", "NIS_BWD_TC")

# kernel families
PACK = ("flow_pack_kernel",)
H_FWD = ("flow_cell_h_kernel", "flow_col_moments_kernel", "flow_h_pack_kernel") + PACK
H_EVAL = ("flow_cell_h_kernel", "flow_h_pack_kernel") + PACK
H_INV = H_FWD + ("flow_inverse_gather_kernel",)
H_INV_EVAL = H_EVAL + ("flow_inverse_gather_kernel",)
WIDE_FWD = ("flow_col_moments_kernel", "flow_wide_pack_kernel", "flow_wide_tc_kernel") + PACK
WIDE_EVAL = ("flow_wide_pack_kernel", "flow_wide_tc_kernel") + PACK
TILED_FWD = ("flow_cell_tiled_kernel", "flow_col_moments_kernel") + PACK
GENERIC = ("flow_fwd_generic_kernel",) + PACK
COOP = ("flow_fwd_coop_kernel",) + PACK
BWD_TC = ("flow_bwd_tail_kernel", "flow_bwd_tc_head_kernel", "flow_bwd_tc_layer_kernel", "flow_bwd_tc_pack_kernel",
          "flow_bwd_tc_reduce_kernel", "flow_tc_pack_kernel") + PACK
BWD_WIDE_CACHED = ("flow_bwd_tail_kernel", "flow_bwd_wide_dgrad_kernel", "flow_bwd_wide_head_kernel",
                   "flow_bwd_wide_pack_kernel", "flow_bwd_wide_reduce_kernel", "flow_bwd_wide_wgrad_kernel",
                   "flow_wide_pack_kernel") + PACK
BWD_WIDE = BWD_WIDE_CACHED + ("flow_wide_tc_kernel",)            # layer passes run again: no activation cache
BWD_GENERIC = ("bwd_reduce_gpart_kernel", "flow_bwd_generic_kernel", "flow_bwd_pack_kernel") + PACK
BWD_COOP = ("flow_bwd_coop_kernel", "flow_bwd_pack_kernel") + PACK

# name, flow, points, mode, knobs, expected (forward, backward, inverse).  The batch thresholds: 256 points for the
# tensor-core kernels, 2048 for the register-tiled one; below them, and with the knobs, the shape-generic kernels run, in one
# cooperative launch while every tile has a resident CTA (2^18 points of cfg2 do not fit: one launch per pass).
ROWS = [
    ("cfg2_eval", CFG2, 4096, "eval", {}, (H_EVAL, BWD_GENERIC, H_INV_EVAL)),
    ("cfg2_train", CFG2, 4096, "train", {}, (H_FWD, BWD_TC, H_INV)),
    ("cfg4_eval", CFG4, 4096, "eval", {}, (H_EVAL, BWD_GENERIC, H_INV_EVAL)),
    ("cfg4_train", CFG4, 4096, "train", {}, (H_FWD, BWD_WIDE, H_INV)),
    ("cfg2_no_tc", CFG2, 4096, "train", {"NIS_TC": "0"}, (TILED_FWD, BWD_GENERIC, GENERIC)),
    ("cfg2_no_tc_no_tiled", CFG2, 4096, "train", {"NIS_TC": "0", "NIS_DISABLE_TILED": "1"}, (COOP, BWD_GENERIC, GENERIC)),
    ("cfg2_no_tc_no_tiled_2p18", CFG2, 1 << 18, "train", {"NIS_TC": "0", "NIS_DISABLE_TILED": "1"},
     (GENERIC, BWD_GENERIC, GENERIC)),
    ("cfg2_no_bwd_tc", CFG2, 4096, "train", {"NIS_BWD_TC": "0"}, (H_FWD, BWD_GENERIC, H_INV)),
    ("cfg2_255", CFG2, 255, "train", {}, (COOP, BWD_GENERIC, GENERIC)),
    ("cfg2_1000", CFG2, 1000, "train", {}, (H_FWD, BWD_TC, H_INV)),
    ("cfg5_small_eval", CFG5_SMALL, 4096, "eval", {}, (WIDE_EVAL, BWD_GENERIC, GENERIC)),
    ("cfg5_small_train", CFG5_SMALL, 4096, "train", {}, (WIDE_FWD, BWD_WIDE_CACHED, GENERIC)),
    ("quad64_20bins", QUAD64_20BINS, 4096, "train", {}, (WIDE_FWD, BWD_WIDE_CACHED, GENERIC)),
    ("readme_2d", README, 2000, "train", {}, (COOP, BWD_COOP, GENERIC)),
    ("affine8d", AFFINE, 4096, "train", {}, (COOP, BWD_GENERIC, GENERIC)),
]


def _kernels(fn):
    """Counter of the library's kernels launched inside fn(), by name without template arguments"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = Counter()
    for e in prof.key_averages():
        m = re.match(r"(?:void )?((?:flow|bwd)_\w+)", e.key)
        if m and e.device_type.name == "CUDA":
            names[m.group(1)] += e.count
    return names


def observe(cfg, B, mode):
    """(forward, backward, inverse): sorted names of the kernels each call launches"""
    torch.manual_seed(3)
    model = make_manager(cfg)._model.cuda()
    model.train(mode == "train")
    gen = torch.Generator().manual_seed(4)
    x = torch.rand(B, cfg["n_flow"], generator=gen, dtype=torch.float64).cuda()
    xj = torch.cat((x, torch.ones(B, 1, dtype=torch.float64, device="cuda")), 1)

    def fwd():
        return model(xj)

    def fwd_bwd():
        (model(xj)[:, -1] ** 2).mean().backward()

    f = _kernels(fwd)
    b = _kernels(fwd_bwd) - f
    i = _kernels(lambda: model.spec().inverse(xj, model.training))
    return tuple(tuple(sorted(k)) for k in (f, b, i))


@pytest.mark.parametrize("name,cfg,B,mode,knobs,expected", ROWS, ids=[r[0] for r in ROWS])
def test_kernel_families(monkeypatch, name, cfg, B, mode, knobs, expected):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    got = observe(cfg, B, mode)
    for what, g, e in zip(("forward", "backward", "inverse"), got, expected):
        assert g == tuple(sorted(e)), "%s %s: %s, expected %s" % (name, what, g, tuple(sorted(e)))
