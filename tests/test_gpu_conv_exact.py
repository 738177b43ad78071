"""Convolution kernels against a float64 oracle, bit for bit, on exact operands (tests/conv_exact.py).

Operands are small integers times powers of two, chosen per case so that every sum of |products| stays below 2^22
granules: every fp32 partial sum is then exact in any order, and the fp32 result must EQUAL the float64 oracle
(torch.equal), element by element.  A norm bound (tests/test_gpu_conv.py, ||err|| / ||ref|| <= 1e-3) cannot see one
wrong row among hundreds of thousands; this can (test_negative_control_one_missing_unit).  Every output and workspace
is filled with NaN before the launch, so a row, a weight or a split-K partial that is never written fails too.

Covered: lg_conv_gemm_tc (forward, dgrad with flipped offsets, power-of-two out_scale, bias) in fp16 and bf16,
lg_conv_wgrad_tc with out_scale, lg_conv_layer_forward (with the batch-norm statistics of its epilogue) and
lg_conv_layer_backward (fp16 gradient scaling by lg_absmax_scale / lg_cast_rows, both powers of two), and the fp32
SIMT kernels on the same plans.  Hand-built plans reach every launch shape of gemm2_shape / wgrad2_shape (the test ids
name them) and the plan edges; the coordinate-derived cases are the tensor-core layers of MinkUNet34.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from lidog_b200 import cabi
from oracle import conv as oc
from oracle import voxel as ov
from tests import conv_exact as cx
from tests.helpers import random_voxels

pytestmark = pytest.mark.gpu

FMTS = {"fp16": (cabi.FMT_FP16, torch.float16), "bf16": (cabi.FMT_BF16, torch.bfloat16)}
REJECTED = (-1, -4)  # LG_ERR_INVALID, LG_ERR_UNSUPPORTED


@pytest.fixture(scope="module")
def sm_count(cuda):
    return cabi.device_info()[0]


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


def _dev_plan(p):
    """lgConvPlan of packed plan arrays (validated again here: nothing unchecked reaches a kernel)."""
    cx.validate_plan(**p)
    nbr = torch.from_numpy(p["nbr"]).cuda()
    out_row = None if p["out_row"] is None else torch.from_numpy(p["out_row"]).cuda()
    mask = torch.from_numpy(p["tile_mask"]).cuda()
    plan = cabi.make_plan(nbr, p["k_stride"], out_row, mask, p["K"], p["n_slots"], p["n_out"], p["n_in"])
    plan._keep = (nbr, out_row, mask)
    return plan


def assert_exact(got, ref, what):
    got = got.detach().cpu().double()
    if torch.equal(got, ref):
        return
    bad = ~(got == ref)
    idx = bad.nonzero()
    diff = (got - ref).abs()[bad]
    raise AssertionError(f"{what}: {int(bad.sum())} of {ref.numel()} elements differ (NaN / unwritten: "
                         f"{int(torch.isnan(got).sum())}); first at {idx[0].tolist()}: got {got[tuple(idx[0])].item()} "
                         f"ref {ref[tuple(idx[0])].item()}; max |diff| {diff.nan_to_num(float('inf')).max().item()}")


def _check_s(abs_sum, exp, what):
    s = cx.granules(abs_sum, exp)
    assert s < cx.S_LIMIT, f"{what}: S = {s} granules: the operand grid is too coarse for an exact comparison"


def _gemm_tc(plan, A16, B16, N, flip, fmt, scale, bias):
    Y = _nan(plan.n_out, N)
    cabi.check(cabi.lib().lg_conv_gemm_tc(C.byref(plan), A16.data_ptr(), A16.shape[1], B16.data_ptr(), N, int(flip),
                                          fmt, cabi.ptr(scale), cabi.ptr(bias), Y.data_ptr(), cabi.stream()),
               "lg_conv_gemm_tc")
    return Y


def _gemm_id(c):
    return f"{c.name}[{cx.gemm_label(c.shape(cx.SM_COUNT_B200))}]".replace(" ", ",")


@pytest.mark.parametrize("case", cx.GEMM_CASES, ids=_gemm_id)
def test_gemm_tc_and_simt_bit_exact(cuda, sm_count, case):
    shape = case.shape(sm_count)
    if case.T:
        assert shape["T"] == case.T, (case.name, shape)
    pl = case.pairs(sm_count)
    p = cx.plan_of_pairs(pl)
    g = torch.Generator().manual_seed(11)
    A = cx.grid_operand(g, (pl.n_in, case.Ck), case.ea)
    B = cx.grid_operand(g, (case.K, case.N, case.Ck), case.eb)  # lg_conv_gemm_tc layout [K][N][Ck]
    ref, ref_abs = cx.gather_gemm(pl, A, B, case.flip)
    _check_s(ref_abs, case.ea + case.eb, case.name)
    bias = cx.grid_operand(g, (case.N,), case.ea + case.eb) if case.bias else None
    scale = 2.0 ** -3 if case.scale else 1.0
    want = ref * scale + (0 if bias is None else bias)
    plan = _dev_plan(p)
    bias_d = None if bias is None else bias.float().cuda()
    scale_d = torch.tensor([scale], dtype=torch.float32, device="cuda") if case.scale else None
    for name, (fmt, dt) in FMTS.items():
        Y = _gemm_tc(plan, A.to(dt).cuda(), B.to(dt).cuda(), case.N, case.flip, fmt, scale_d, bias_d)
        assert_exact(Y, want, f"{case.name} lg_conv_gemm_tc {name} ({cx.gemm_label(shape)})")
    # fp32 SIMT kernel, same plan: W stored [K][N][Ck] = w_transposed
    Y = _nan(pl.n_out, case.N)
    A32, B32 = A.float().cuda(), B.float().cuda()  # held: a freed temporary's block would be reused by the next one
    cabi.check(cabi.lib().lg_conv_gemm_simt(C.byref(plan), A32.data_ptr(), case.Ck, B32.data_ptr(), case.N, 1,
                                            int(case.flip), cabi.ptr(bias_d), Y.data_ptr(), cabi.stream()),
               "lg_conv_gemm_simt")
    assert_exact(Y, ref + (0 if bias is None else bias), f"{case.name} lg_conv_gemm_simt")


def _wgrad_id(c):
    return f"{c.name}[{cx.wgrad_label(c.shape(), c.tiles)}]".replace(" ", ",")


@pytest.mark.parametrize("case", cx.WGRAD_CASES, ids=_wgrad_id)
def test_wgrad_tc_and_simt_bit_exact(cuda, case):
    L = cabi.lib()
    pl = case.pairs()
    p = cx.plan_of_pairs(pl)
    g = torch.Generator().manual_seed(12)
    X = cx.grid_operand(g, (pl.n_in, case.Cin), case.ea)
    dY = cx.grid_operand(g, (pl.n_out, case.Cout), case.eb)
    ref, ref_abs = cx.wgrad(pl, X, dY)
    _check_s(ref_abs, case.ea + case.eb, case.name)
    plan = _dev_plan(p)
    scale = torch.tensor([0.25], dtype=torch.float32, device="cuda")
    for name, (fmt, dt) in FMTS.items():
        ws_bytes = L.lg_conv_wgrad_tc_workspace(C.byref(plan), case.Cin, case.Cout)
        ws = _nan(ws_bytes // 4)  # split-K partials: a chunk that never writes its partial leaves NaN in dW
        dW = _nan(case.K, case.Cin, case.Cout)
        X16, dY16 = X.to(dt).cuda(), dY.to(dt).cuda()
        cabi.check(L.lg_conv_wgrad_tc(C.byref(plan), X16.data_ptr(), case.Cin, dY16.data_ptr(), case.Cout, fmt,
                                      scale.data_ptr(), dW.data_ptr(), ws.data_ptr(), ws_bytes, cabi.stream()),
                   "lg_conv_wgrad_tc")
        assert_exact(dW, ref * 0.25,
                     f"{case.name} lg_conv_wgrad_tc {name} ({cx.wgrad_label(case.shape(), case.tiles)})")
    ws_bytes = L.lg_conv_wgrad_workspace(C.byref(plan), case.Cin, case.Cout)
    ws = _nan(max(ws_bytes // 4, 1))
    dW = _nan(case.K, case.Cin, case.Cout)
    X32, dY32 = X.float().cuda(), dY.float().cuda()
    cabi.check(L.lg_conv_wgrad_simt(C.byref(plan), X32.data_ptr(), case.Cin, dY32.data_ptr(), case.Cout, dW.data_ptr(),
                                    ws.data_ptr(), ws_bytes, cabi.stream()), "lg_conv_wgrad_simt")
    assert_exact(dW, ref, f"{case.name} lg_conv_wgrad_simt")


# ------------------------------------------------------------------------------------------------ MinkUNet34 layers
@pytest.fixture(scope="module")
def cloud(cuda):
    import MinkowskiEngine as ME
    coords = random_voxels(np.random.default_rng(0), 9000, span=30)
    base = ME.SparseTensor(coordinates=torch.from_numpy(coords).cuda(), features=torch.ones(len(coords), 1).cuda())
    cm = base.coordinate_manager
    return cm, {ts: cm.get_coords(ts).cpu().numpy() for ts in (1, 2, 4, 8, 16)}


def _layer(cm, cc, kind, ts, order):
    """(forward, dgrad, wgrad plans, flip of dgrad) as MinkowskiConvolutionBase._plans builds them, the oracle's
    pair lists from oracle.voxel, n_in, n_out."""
    sfx = "_sorted" if order == "sorted" else ""
    if kind == "same":
        p = cm.plan("same" + sfx, ts, ts, 3)
        return (p, p, p, 1), ov.kernel_map(cc[ts], cc[ts], 3, ts), len(cc[ts]), len(cc[ts])
    if kind == "down":
        down = cm.plan("down" + sfx, ts, 2 * ts, 2)
        return ((down, cm.plan("up", 2 * ts, ts, 2), down, 0), ov.kernel_map(cc[ts], cc[2 * ts], 2, ts),
                len(cc[ts]), len(cc[2 * ts]))
    if kind == "up":
        up = cm.plan("up", ts, ts // 2, 2)
        return ((up, cm.plan("down" + sfx, ts // 2, ts, 2), up, 0),
                ov.transposed_kernel_map(cc[ts // 2], cc[ts], 2, ts // 2), len(cc[ts]), len(cc[ts // 2]))
    p = cm.plan("identity", ts, ts, 1)
    r = np.arange(len(cc[ts]))
    return (p, p, p, 0), [(r, r)], len(cc[ts]), len(cc[ts])


# Natural-order plans exist for the 3x3x3 and stride-2 layers; the "up" and 1x1 plans have one order.  The sorted plans
# run in fp16, the natural ones in bf16.
LAYER_CASES = [(s, "sorted") for s in cx.minkunet34_conv_shapes()] + \
    [(s, "natural") for s in cx.minkunet34_conv_shapes() if s[0] in ("same", "down")]


@pytest.mark.parametrize("shape,order", LAYER_CASES, ids=lambda v: "-".join(map(str, v)) if isinstance(v, tuple) else v)
def test_layer_forward_backward_bit_exact(cuda, cloud, shape, order):
    kind, ts, ksize, cin, cout = shape
    cm, cc = cloud
    (pf, pd, pw, flip), maps, n_in, n_out = _layer(cm, cc, kind, ts, order)
    fmt, dt = FMTS["fp16" if order == "sorted" else "bf16"]
    L = cabi.lib()
    K = ksize ** 3
    g = torch.Generator().manual_seed(13)
    ex, ew, ed = 3, 6, 4
    x = cx.grid_operand(g, (n_in, cin), ex)
    W = cx.grid_operand(g, (K, cin, cout), ew)
    dY = cx.grid_operand(g, (n_out, cout), ed)
    y_ref = oc.conv_forward(x, W, maps, n_out)
    _check_s(oc.conv_forward(x.abs(), W.abs(), maps, n_out), ex + ew, "forward")
    dx_ref = oc.conv_dgrad(dY, W, maps, n_in)
    _check_s(oc.conv_dgrad(dY.abs(), W.abs(), maps, n_in), ed + ew, "dgrad")
    dw_ref = oc.conv_wgrad(x, dY, maps, K)
    _check_s(oc.conv_wgrad(x.abs(), dY.abs(), maps, K), ex + ed, "wgrad")

    x16 = x.to(dt).cuda()
    w16 = torch.empty((K, cin, cout), dtype=dt, device="cuda")
    w16t = torch.empty((K, cout, cin), dtype=dt, device="cuda")
    Y = _nan(n_out, cout)
    stats = _nan(4 * pf.n_tiles, 2 * cout)
    W32 = W.float().cuda()
    cabi.check(L.lg_conv_layer_forward(pf.cref, x16.data_ptr(), cin, W32.data_ptr(), cout, w16.data_ptr(),
                                       w16t.data_ptr(), 1, fmt, None, Y.data_ptr(), stats.data_ptr(), cabi.stream()),
               "lg_conv_layer_forward")
    assert_exact(Y, y_ref, "lg_conv_layer_forward Y")
    # Epilogue statistics: per (tile, epilogue warp) = 32 slots, the column sums and sums of squares of Y.  The squares
    # of grid values need twice the bits, so neither is exact in fp32 in every order: element-wise bound
    # 32 * 2^-24 * sum |terms| (32 terms of one warp's rows, each add rounding by at most 2^-24 relative).
    rows = (torch.arange(pf.n_slots) if pf.out_row is None else pf.out_row.cpu().long())
    valid = (rows >= 0) & (rows < n_out)
    yr = torch.where(valid[:, None], y_ref[rows.clamp(0, max(n_out - 1, 0))], torch.zeros((), dtype=torch.float64))
    yr = yr.view(-1, 32, cout)
    st = stats.cpu().double()
    for got, terms, what in ((st[:, :cout], yr, "column sums"), (st[:, cout:], yr * yr, "sums of squares")):
        bound = 32 * 2.0 ** -24 * terms.abs().sum(1)
        err = (got - terms.sum(1)).abs()
        assert not torch.isnan(got).any(), f"stat_partials {what}: unwritten rows"
        assert (err <= bound).all(), f"stat_partials {what}: max excess {(err - bound).max().item()}"

    dY32 = dY.float().cuda()
    scale = torch.empty(4, dtype=torch.float32, device="cuda")
    cabi.check(L.lg_absmax_scale(dY32.data_ptr(), dY32.numel(), scale.data_ptr(), cabi.stream()), "lg_absmax_scale")
    dY16 = torch.empty((n_out, cout), dtype=dt, device="cuda")
    cabi.check(L.lg_cast_rows(dY32.data_ptr(), dY16.data_ptr(), dY32.numel(), fmt, scale.data_ptr(), cabi.stream()),
               "lg_cast_rows")
    s = scale.cpu()
    assert s[0] * s[1] == 1 and torch.frexp(s[:1]).mantissa.item() == 0.5  # a power of two and its inverse
    dX = _nan(n_in, cin)
    dW = _nan(K, cin, cout)
    cabi.check(L.lg_conv_layer_backward(pd.cref, pw.cref, flip, x16.data_ptr(), cin, dY16.data_ptr(), cout,
                                        w16.data_ptr(), fmt, scale.data_ptr() + 4, dX.data_ptr(), dW.data_ptr(),
                                        cabi.stream()), "lg_conv_layer_backward")
    assert_exact(dX, dx_ref, "lg_conv_layer_backward dX")
    assert_exact(dW, dw_ref, "lg_conv_layer_backward dW")


# ------------------------------------------------------------------------------------------------ negative control
def test_negative_control_one_missing_unit(cuda):
    """Clear one mask bit of one tile in the plan the kernel gets (the plan stays valid) and keep the oracle: the exact
    comparison fails, while the relative-norm bound of tests/test_gpu_conv.py (1e-3) would have passed."""
    case = cx.GemmCase("negative_control", 64, 64, 8, tiles=200)
    pl = case.pairs(cx.SM_COUNT_B200)
    rows = pl.result_rows()
    j = int(np.flatnonzero((rows >= 0) & (pl.slot // cx.TILE > 3))[0])
    k, t = int(pl.k[j]), int(pl.slot[j] // cx.TILE)
    # the unit (tile t, offset k) keeps this one pair, gathering an extra input row with one nonzero element
    drop = (pl.k == k) & (pl.slot // cx.TILE == t) & (np.arange(pl.k.size) != j)
    pl.k, pl.slot, pl.inp = pl.k[~drop], pl.slot[~drop], pl.inp[~drop]
    j = int(np.flatnonzero((pl.k == k) & (pl.slot // cx.TILE == t))[0])
    pl.inp[j] = pl.n_in
    pl.n_in += 1
    g = torch.Generator().manual_seed(14)
    A = cx.grid_operand(g, (pl.n_in, case.Ck), case.ea)
    A[-1] = 0
    A[-1, 0] = 2.0 ** -case.ea
    B = cx.grid_operand(g, (case.K, case.N, case.Ck), case.eb)
    B[k, 0, 0] = 2.0 ** -case.eb
    ref, _ = cx.gather_gemm(pl, A, B, False)
    p = cx.plan_of_pairs(pl)
    fmt, dt = FMTS["fp16"]
    A16, B16 = A.to(dt).cuda(), B.to(dt).cuda()
    assert_exact(_gemm_tc(_dev_plan(p), A16, B16, case.N, False, fmt, None, None), ref, "intact plan")
    mask = p["tile_mask"].copy()
    mask[t, k // 32] &= ~np.int32(1 << (k % 32))
    Y = _gemm_tc(_dev_plan({**p, "tile_mask": mask}), A16, B16, case.N, False, fmt, None, None).cpu().double()
    assert not torch.equal(Y, ref)
    assert int((Y != ref).any(1).sum()) == 1  # exactly the one result row of the dropped pair
    assert float((Y - ref).norm() / ref.norm()) <= 1e-3


# ------------------------------------------------------------------------------------------------ rejected inputs
def _tiny_plan(K, tiles=1):
    pl = cx.make_pairs(np.random.default_rng(5), K, tiles, edges=False, masks="random" if K <= 32 else "hi_lo")
    return _dev_plan(cx.plan_of_pairs(pl)), pl


def test_host_rejects_unsupported_shapes_before_launch(cuda):
    L = cabi.lib()
    fmt, dt = FMTS["fp16"]
    plan, pl = _tiny_plan(8)
    for Ck, N in ((64, 400), (64, 336), (48, 64)):  # column blocks of 200 / 168 columns; Ck not a multiple of 32
        A = torch.zeros((pl.n_in, Ck), dtype=dt, device="cuda")
        B = torch.zeros((8, N, Ck), dtype=dt, device="cuda")
        Y = _nan(pl.n_out, N)
        rc = L.lg_conv_gemm_tc(C.byref(plan), A.data_ptr(), Ck, B.data_ptr(), N, 0, fmt, None, None, Y.data_ptr(),
                               cabi.stream())
        assert rc in REJECTED, (Ck, N, rc)
        assert torch.isnan(Y).all()
    plan125, pl125 = _tiny_plan(125)
    for K_plan, pln, Cin, Cout in ((125, plan125, 32, 32), (8, plan, 32, 288)):
        X = torch.zeros((pln.n_in, Cin), dtype=dt, device="cuda")
        dY = torch.zeros((pln.n_out, Cout), dtype=dt, device="cuda")
        ws_bytes = max(L.lg_conv_wgrad_tc_workspace(C.byref(pln), Cin, Cout), 4 * K_plan * Cin * Cout + 256)
        ws = _nan(ws_bytes // 4)
        dW = _nan(K_plan, Cin, Cout)
        rc = L.lg_conv_wgrad_tc(C.byref(pln), X.data_ptr(), Cin, dY.data_ptr(), Cout, fmt, None, dW.data_ptr(),
                                ws.data_ptr(), ws_bytes, cabi.stream())
        assert rc in REJECTED, (K_plan, Cout, rc)
        assert torch.isnan(dW).all()
