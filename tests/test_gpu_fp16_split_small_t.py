"""flow_tc_h.cu with few transformed dimensions per PWLin cell: an output layer of one MMA block (T = 1, 2) or a last
block without its second dimension (T = 3), with the next cell's column moments fused into the final pass (P <= 4)
and a one-column pass-through (P = 1)."""
import pytest

import test_gpu_flow as tgf

pytestmark = pytest.mark.gpu

SMALL_T = [
    dict(name="lin5d_T1", kind="lin", n_flow=5, n_pass_through=4, n_cells=5, n_bins=32, NN=[64] * 3, roll_step=1, B=5000),
    dict(name="lin6d_T2", kind="lin", n_flow=6, n_pass_through=4, n_cells=4, n_bins=32, NN=[64] * 3, roll_step=2, B=5000),
    dict(name="lin7d_T3", kind="lin", n_flow=7, n_pass_through=4, n_cells=5, n_bins=32, NN=[64] * 3, roll_step=3, B=5000),
    dict(name="lin4d_T3_P1", kind="lin", n_flow=4, n_pass_through=1, n_cells=4, n_bins=32, NN=[64] * 3, roll_step=1, B=5000),
]


@pytest.mark.parametrize("cfg", SMALL_T, ids=[c["name"] for c in SMALL_T])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_pwlin_with_few_transformed_dimensions(cfg, mode):
    tgf.test_forward_matches_oracle_at_size(cfg, mode)
