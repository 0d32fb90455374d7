"""GPU parity of the fused flow forward (through FlowSequential -> nis_flow_forward) against
(a) the golden vectors dumped from the reference and (b) the oracle at larger sizes."""
import numpy as np
import pytest
import torch

from conftest import FLOW_CASES
from gpu_util import compare_flow, make_manager, oracle_layers
from oracle import flow as oflow

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("case", FLOW_CASES)
@pytest.mark.parametrize("mode", ["eval", "train"])
@pytest.mark.parametrize("io", [torch.float64, torch.float32])
def test_forward_matches_reference_golden(golden, case, mode, io):
    g = golden("flow_" + case)
    NF = make_manager(g.meta)
    model = NF._model
    model.load_state_dict(g.state_dict())
    model.train(mode == "train")
    xj = g.t("xj").to(io).cuda()
    XJ, bins = model.forward_with_bins(xj)
    assert XJ.dtype == io and XJ.shape == xj.shape
    if g.meta["kind"] == "affine":           # no bins: the kernel reports 0 for every transformed dimension
        T = g.meta["n_flow"] - g.meta["n_pass_through"]
        ref_bins = [np.zeros((xj.shape[0], T), np.int32) for _ in range(model.spec().n_cells)]
    else:
        ref_bins = [g["%s/bins/%d" % (mode, i)] for i in range(model.spec().n_cells)]
    edges = []                              # distances to the nearest bin edge, from the oracle (== reference to 1e-12)
    with torch.no_grad():
        oflow.flow_forward(oracle_layers(g.meta), g.state_dict(), g.t("xj"), g.meta["kind"], g.meta["n_bins"],
                           train=(mode == "train"), edges=edges)
    compare_flow(XJ.cpu(), bins.cpu(), g.t(mode + "/XJ"), ref_bins, "%s/%s" % (case, mode),
                 ref_edges=[e.numpy() for e in edges] if edges else None)
    if mode == "train":                      # running statistics updated like torch BatchNorm1d
        sd = model.state_dict()
        for k in g.keys("train/stats/"):
            name = k[len("train/stats/"):]
            ref = g.t(k)
            if name.endswith("num_batches_tracked"):
                assert int(sd[name]) == int(ref)
            else:
                assert torch.allclose(sd[name].double().cpu(), ref, rtol=2e-5, atol=1e-6), name


@pytest.mark.parametrize("case", ["quad2d", "lin4d", "quad8d_small"])
def test_autograd_entry_equals_plain_forward_and_accepts_d_columns(golden, case):
    g = golden("flow_" + case)
    NF = make_manager(g.meta)
    model = NF._model
    model.load_state_dict(g.state_dict())
    model.eval()
    xj = g.t("xj").cuda()
    a = model(xj)
    b, _ = model.forward_with_bins(xj)
    assert torch.equal(a, b)
    x_only = xj[:, :-1].contiguous()
    c, _ = model.forward_with_bins(x_only)                       # J = 1 implied
    assert torch.allclose(c[:, -1] * xj[:, -1], a[:, -1], rtol=1e-6)
    assert torch.equal(c[:, :-1], a[:, :-1])


BIG = [
    dict(name="cfg2", kind="lin", n_flow=8, n_pass_through=4, n_cells=6, n_bins=32, NN=[64] * 3, roll_step=4, B=1 << 15),
    dict(name="cfg4", kind="quad", n_flow=8, n_cells=6, n_bins=32, NN=[64] * 3, B=1 << 14),
    dict(name="cfg1", kind="quad", n_flow=2, n_cells=2, n_bins=4, NN=[3] * 3, B=10000),
    dict(name="cfg5_small", kind="quad", n_flow=16, n_cells=8, n_bins=64, NN=[256] * 2, B=1 << 11),
]


@pytest.mark.parametrize("cfg", BIG, ids=[c["name"] for c in BIG])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_forward_matches_oracle_at_size(cfg, mode, max_log_j=None, mutate_sd=None):
    torch.manual_seed(5)
    NF = make_manager(cfg)
    model = NF._model
    cells, out_perm = oflow.compile_layers(oracle_layers(cfg), cfg["n_flow"])
    sd = oflow.init_state_dict(cells, cfg["n_flow"], cfg["kind"], cfg["n_bins"], cfg["NN"], seed=7,
                               dtype=torch.float32, bn_jitter=0.2)
    if mutate_sd is not None:
        mutate_sd(sd)
    model.load_state_dict(sd)
    model.train(mode == "train")
    gen = torch.Generator().manual_seed(2026)
    x = torch.rand(cfg["B"], cfg["n_flow"], generator=gen, dtype=torch.float32).double()
    xj = NF.format_input(x, torch.device("cuda"))
    XJ, bins = model.forward_with_bins(xj)
    sd64 = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    edges, cond = [], []
    with torch.no_grad():
        ref, ref_bins = oflow.flow_forward(oracle_layers(cfg), sd64, xj.cpu(), cfg["kind"], cfg["n_bins"],
                                           train=(mode == "train"), edges=edges, clamp_bins=True, cond=cond)
        sd32 = {k: (v.float() if v.dtype.is_floating_point else v) for k, v in sd.items()}
        ref32, _ = oflow.flow_forward(oracle_layers(cfg), sd32, xj.cpu().float(), cfg["kind"], cfg["n_bins"],
                                      train=(mode == "train"), clamp_bins=True)
    compare_flow(XJ.cpu(), bins.cpu(), ref, [b.numpy() for b in ref_bins], "%s/%s" % (cfg["name"], mode),
                 fp32_yardstick=ref32, ref_edges=[e.numpy() for e in edges], max_log_j=max_log_j,
                 ref_cond=[c.numpy() for c in cond])


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_bench_configuration_against_the_oracle_at_a_million_points(mode):
    """cfg2 (the bench workload) at 2^20 points, every point against the float64 oracle: bins (each difference
    proven to sit on an edge), transformed points, and the log-Jacobian with its MAXIMUM bounded (printed)."""
    test_forward_matches_oracle_at_size(dict(BIG[0], B=1 << 20), mode, max_log_j=1e-4)


# cfg2, cfg4, cfg5_small, and two width-64 flows whose fp16-split launch sequences differ from cfg2's and cfg4's: PWLin at
# depth 2 with six pass-through columns (no recomputed last layer, column moments in a launch of their own for every cell),
# and PWQuad with one hidden layer (the final pass starts from the state)
FAMILY = [BIG[0], BIG[1], BIG[3],
          dict(name="lin8d_depth2_6pass", kind="lin", n_flow=8, n_pass_through=6, n_cells=4, n_bins=32, NN=[64] * 2,
               roll_step=3, B=1 << 13),
          dict(name="quad8d_1layer", kind="quad", n_flow=8, n_cells=4, n_bins=32, NN=[64], B=1 << 13)]


@pytest.mark.parametrize("backend", ["tcgen05", "fp32_tiled_4x8", "generic"])
@pytest.mark.parametrize("mode", ["eval", "train"])
@pytest.mark.parametrize("cfg", FAMILY, ids=[c["name"] for c in FAMILY])
def test_every_kernel_family_agrees_with_the_oracle(monkeypatch, backend, mode, cfg):
    """The width-64 flows with 32 bins are served by the fp16-split tcgen05 kernel by default, the 256-wide cfg5 by the
    streamed-weights one (flow_wide.cu); the FP32-pipe register-tiled kernel and the shape-generic kernel stay
    selectable (library test knobs) and must meet the same parity bar."""
    if cfg["NN"][0] != 64 and backend.startswith("fp32_tiled"):
        pytest.skip("the register-tiled FP32 kernels are width-64 only")
    env = {"tcgen05": {}, "fp32_tiled_4x8": {"NIS_TC": "0"}, "generic": {"NIS_TC": "0", "NIS_DISABLE_TILED": "1"}}[backend]
    for k in ("NIS_TC", "NIS_DISABLE_TILED"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    test_forward_matches_oracle_at_size(cfg, mode)
    # ragged batch (not a multiple of any tile size) through the same kernels
    test_forward_matches_oracle_at_size(dict(cfg, B=(1 << 13) + 77), mode)


def test_flow_is_a_bijection_of_the_unit_cube_at_full_size():
    """Size-independent properties at cfg2's full batch (2^22 points): <J> = 1 within Monte Carlo error,
    outputs stay in [0,1], pass-through columns of the last cell are bit-identical to its input."""
    torch.manual_seed(11)
    cfg = BIG[0]
    NF = make_manager(cfg)
    model = NF._model.eval()
    B = 1 << 22
    x = torch.rand(B, 8, device="cuda", dtype=torch.float32)
    XJ = model(x)
    J = XJ[:, -1].double()
    assert abs(float(J.mean()) - 1.0) < 6 * float(J.std()) / np.sqrt(B)
    assert float(XJ[:, :-1].min()) >= 0.0 and float(XJ[:, :-1].max()) <= 1.0 + 1e-6
    # determinism: same input, same bits
    assert torch.equal(model(x), XJ)


WIDE = [
    dict(name="wide_lin128", kind="lin", n_flow=8, n_pass_through=4, n_cells=4, n_bins=48, NN=[128] * 3, roll_step=4, B=3000),
    dict(name="wide_quad192", kind="quad", n_flow=6, n_cells=6, n_bins=20, NN=[192] * 2, B=2500),
    dict(name="quad64_20bins", kind="quad", n_flow=8, n_cells=6, n_bins=20, NN=[64] * 3, B=3000),
    dict(name="wide_quad256_deep", kind="quad", n_flow=16, n_cells=8, n_bins=64, NN=[256] * 4, B=1400),
]


@pytest.mark.parametrize("cfg", WIDE, ids=[c["name"] for c in WIDE])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_streamed_weight_kernel_shapes(cfg, mode):
    """flow_wide.cu beyond cfg5_small: width 128 (one round), 192 (one round of N = 192), 256 x 4 layers (two rounds
    per hidden layer), PWLin and PWQuad, bin counts that are not multiples of 16, ragged last tile."""
    test_forward_matches_oracle_at_size(cfg, mode)


AFFINE = [
    dict(name="affine8d_wide", kind="affine", n_flow=8, n_pass_through=4, n_cells=4, n_bins=1, NN=[64] * 2, roll_step=4, B=5000),
    dict(name="affine3d", kind="affine", n_flow=3, n_pass_through=1, n_cells=5, n_bins=1, NN=[8, 8, 8], roll_step=1, B=777),
]


@pytest.mark.parametrize("cfg", AFFINE, ids=[c["name"] for c in AFFINE])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_affine_coupling_flow_matches_oracle_at_size(cfg, mode):
    """AffineCoupling / AffineManager (coupling_cells.py:6-70, manager.py:411-453; SURVEY 8 f4) on the shape-generic kernels:
    y = atan(20 e^{Z0} x + relu(Z1)) / (pi/2), 1/(pi/2) once per cell in the Jacobian, hidden layers WITH bias (folded into
    the running mean the kernels see), Reshape(2, T) row order of the output layer; a 64-wide conditioner must not be
    taken by the tensor-core paths."""
    test_forward_matches_oracle_at_size(cfg, mode)


MANY_PASS_THROUGH = [
    dict(name="lin13d_9pass", kind="lin", n_flow=13, n_pass_through=9, n_cells=4, n_bins=32, NN=[64] * 3, roll_step=3, B=2700),
    dict(name="lin20d_16pass", kind="lin", n_flow=20, n_pass_through=16, n_cells=3, n_bins=32, NN=[64] * 2, roll_step=7, B=1500),
    dict(name="quad18d", kind="quad", n_flow=18, n_cells=5, n_bins=32, NN=[64] * 3, B=1300),
    dict(name="lin6d_1layer", kind="lin", n_flow=6, n_pass_through=3, n_cells=4, n_bins=32, NN=[64], roll_step=2, B=2100),
]


@pytest.mark.parametrize("cfg", MANY_PASS_THROUGH, ids=[c["name"] for c in MANY_PASS_THROUGH])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_fp16_split_kernel_pass_through_counts(cfg, mode):
    """flow_tc_h.cu with 9 .. 16 pass-through columns: the first linear layer is one K = 16 tensor-core step whatever P
    is, and beyond 8 columns the statistics of BN_1 come from a layer pass of their own (the one-pass column moments
    stop at P = 8); a one-hidden-layer conditioner (no chained hidden layer at all)."""
    test_forward_matches_oracle_at_size(cfg, mode)


@pytest.mark.parametrize("which", [0, 1, 3], ids=["cfg2", "cfg4", "cfg5_small"])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_tensor_core_kernels_at_small_batches(which, mode):
    """The tensor-core kernels take over from 256 points (a training minibatch of a few hundred points is common in
    the reference's examples): three tiles, the last one ragged, a grid of two or three CTAs."""
    test_forward_matches_oracle_at_size(dict(BIG[which], B=300), mode)


INV = [
    dict(name="lin8d", kind="lin", n_flow=8, n_pass_through=4, n_cells=6, n_bins=32, NN=[64] * 3, roll_step=4, B=3000),
    dict(name="quad8d", kind="quad", n_flow=8, n_cells=6, n_bins=32, NN=[64] * 3, B=3000),
    dict(name="quad2d", kind="quad", n_flow=2, n_cells=2, n_bins=4, NN=[3] * 3, B=2000),
    dict(name="quad9d_extra", kind="quad", n_flow=9, n_cells=10, n_bins=6, NN=[16, 16], B=777),
    dict(name="lin5d", kind="lin", n_flow=5, n_pass_through=1, n_cells=4, n_bins=7, NN=[12], roll_step=2, B=1025),
    dict(name="affine6d", kind="affine", n_flow=6, n_pass_through=3, n_cells=4, n_bins=1, NN=[16], roll_step=2, B=1500),
]


@pytest.mark.parametrize("cfg", INV, ids=[c["name"] for c in INV])
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_inverse_flow(cfg, mode):
    """SURVEY 8 f4: FlowSequential.inverse (nis_flow_inverse).  (a) against the float64 inverse of the oracle on the same
    points: same bins (except on an edge), latent points and log-Jacobian within the forward's bars scaled by the local
    stretch; (b) round trip through the CUDA forward (tensor-core kernels where they apply): inverse(forward(x)) = x,
    Jacobian 1."""
    torch.manual_seed(9)
    NF = make_manager(cfg)
    model = NF._model
    cells, out_perm = oflow.compile_layers(oracle_layers(cfg), cfg["n_flow"])
    sd = oflow.init_state_dict(cells, cfg["n_flow"], cfg["kind"], cfg["n_bins"], cfg["NN"], seed=11,
                               dtype=torch.float32, bn_jitter=0.2)
    model.load_state_dict(sd)
    model.train(mode == "train")
    sd64 = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    gen = torch.Generator().manual_seed(77)
    y = (0.002 + 0.996 * torch.rand(cfg["B"], cfg["n_flow"], generator=gen, dtype=torch.float32)).double()
    yj = torch.cat((y, torch.ones(cfg["B"], 1, dtype=torch.float64)), 1)
    X, bins = model.spec().inverse(yj.cuda(), model.training, want_bins=True)
    with torch.no_grad():
        ref, ref_bins = oflow.flow_inverse(oracle_layers(cfg), sd64, yj, cfg["kind"], cfg["n_bins"], train=(mode == "train"))
    X, bins = X.cpu(), bins.cpu()
    same = torch.ones(cfg["B"], dtype=torch.bool)
    for c, rb in enumerate(ref_bins):
        same &= (bins[c, :, :rb.shape[1]].long() == rb).all(1)
    assert float(same.float().mean()) > 0.995, float(same.float().mean())
    if cfg["kind"] == "affine":
        # The affine flow maps the unit cube INTO a subset of itself, and inverting the atan squashing multiplies an error
        # by (pi/2)(1 + v^2) / s0 (up to ~1e3) in EVERY cell: for a y outside the image the next conditioner sees
        # pass-through values like -30 or 200, and even on image points two float32 evaluations of a four-cell inverse agree
        # only to ~1e-2.  The kernel is therefore checked in the well-conditioned direction, on image points (y = forward(x)
        # from the oracle): the float64 FORWARD of what the kernel returned - points and Jacobian column - must give y back;
        # then through the CUDA round trip below.
        xs = (0.002 + 0.996 * torch.rand(cfg["B"], cfg["n_flow"], generator=gen, dtype=torch.float32)).double()
        with torch.no_grad():
            img, _ = oflow.flow_forward(oracle_layers(cfg), sd64, torch.cat((xs, torch.ones(cfg["B"], 1, dtype=torch.float64)), 1),
                                        cfg["kind"], cfg["n_bins"], train=(mode == "train"))
        img32 = img.float().double()
        Xi = model.spec().inverse(img32.cuda(), model.training)[0].cpu().double()
        with torch.no_grad():
            fw, _ = oflow.flow_forward(oracle_layers(cfg), sd64, Xi, cfg["kind"], cfg["n_bins"], train=(mode == "train"))
        dp = (fw[:, :-1] - img32[:, :-1]).abs().max(1).values
        assert float(torch.quantile(dp, 0.999)) < 2e-5, (float(torch.quantile(dp, 0.999)), float(dp.max()))
        lj = (torch.log(fw[:, -1]) - torch.log(img32[:, -1])).abs()
        assert float(torch.quantile(lj, 0.99)) < 2e-4 and float(lj.median()) < 2e-5, (float(lj.median()), float(lj.max()))
    else:
        # |dx| = |dy| / density: compare in units of the local stretch (the Jacobian column holds 1 / prod density)
        stretch = ref[:, -1].clamp_min(1.0)
        err = ((X[:, :-1] - ref[:, :-1]).abs().max(1).values / stretch)[same]
        assert float(err.max()) < 2e-5, float(err.max())
        lj = (torch.log(X[:, -1]) - torch.log(ref[:, -1])).abs()[same]
        assert float(torch.quantile(lj, 0.99)) < 1e-4 and float(lj.median()) < 1e-5, (float(lj.median()), float(lj.max()))
    # round trip through the CUDA forward
    x = (0.002 + 0.996 * torch.rand(cfg["B"], cfg["n_flow"], generator=gen, dtype=torch.float32)).double().cuda()
    with torch.no_grad():
        Y = model(NF.format_input(x, torch.device("cuda")))
        back = model.inverse(Y)
    rt = (back[:, :-1] - x).abs().max(1).values * Y[:, -1].clamp_max(1.0)      # stretch of the inverse = 1 / J
    assert float(torch.quantile(rt, 0.999)) < 2e-5, float(rt.max())
    if cfg["kind"] != "affine":              # (affine: the Jacobian along a path that float32 rounding has moved by ~1e-2 in latent
        assert float(torch.quantile((torch.log(back[:, -1])).abs(), 0.99)) < 2e-4      # space is not 1 to 2e-4; see above)
