"""CPU checks of the exact-operand convolution tests (tests/conv_exact.py): plan packer and validator, float64 oracle,
operand grid, and coverage of the launch shapes the GPU cases reach."""
import numpy as np
import pytest
import torch

from oracle import conv as oc
from tests import conv_exact as cx

SM = cx.SM_COUNT_B200


def _pairs_of_plan(p):
    """Unpack a packed plan back into its (k, slot, input) triples (the inverse of pack_plan)."""
    nbr, mask = p["nbr"], p["tile_mask"].view(np.uint32)
    out = []
    for k in range(p["K"]):
        bit = ((mask[:, k // 32] >> np.uint32(k % 32)) & 1).astype(bool)
        row = nbr if p["k_stride"] == 0 else nbr[k]
        slots = np.flatnonzero(np.repeat(bit, cx.TILE) & (row >= 0))
        out += [(k, s, int(row[s])) for s in slots]
    return sorted(out)


@pytest.mark.parametrize("case", cx.GEMM_CASES + cx.WGRAD_CASES, ids=lambda c: c.name)
def test_packer_round_trips_and_plan_is_valid(case):
    pl = case.pairs(SM) if isinstance(case, cx.GemmCase) else case.pairs()
    p = cx.plan_of_pairs(pl)  # validates
    assert _pairs_of_plan(p) == sorted(zip(pl.k.tolist(), pl.slot.tolist(), pl.inp.tolist()))
    if pl.extra_mask is not None and pl.n_tiles >= 3:
        # the plan edges are present: a masked tile whose slots are all -1, an empty tile, a same-row tile
        m = p["tile_mask"].view(np.uint32)
        assert m[1].any() and not m[2].any()
        t0 = pl.slot < cx.TILE
        assert any(np.unique(pl.inp[t0 & (pl.k == k)]).size == 1 and (t0 & (pl.k == k)).sum() == cx.TILE
                   for k in range(pl.K))


def test_validator_rejects_unsafe_plans():
    pl = cx.make_pairs(np.random.default_rng(1), 8, 4)
    good = cx.plan_of_pairs(pl)
    bad = [dict(nbr=np.where(good["nbr"] >= 0, good["n_in"], -1).astype(np.int32)),
           dict(nbr=np.full_like(good["nbr"], -2)),
           dict(out_row=np.full(good["n_slots"], good["n_out"], np.int32)),
           dict(out_row=np.zeros(good["n_slots"], np.int32)),  # every slot writes row 0
           dict(n_slots=good["n_slots"] - 1)]
    m = good["tile_mask"].copy()
    m[0, 0] |= np.int32(1 << 9)  # bit 9 of an 8-offset plan
    bad.append(dict(tile_mask=m))
    for override in bad:
        with pytest.raises(AssertionError):
            cx.validate_plan(**{**good, **override})


def test_oracle_equals_reference_sparse_conv_function():
    """The pair-list oracle computes what oracle/conv.py's SparseConvFunction computes on the same pairs."""
    pl = cx.make_pairs(np.random.default_rng(2), 8, 6, n_out=6 * 128 - 9, order="perm")
    g = torch.Generator().manual_seed(0)
    Ck, N = 32, 48
    x = cx.grid_operand(g, (pl.n_in, Ck), 3).requires_grad_(True)
    w = cx.grid_operand(g, (pl.K, Ck, N), 6).requires_grad_(True)
    rows = pl.result_rows()
    keep = rows >= 0
    maps = [(pl.inp[keep & (pl.k == k)], rows[keep & (pl.k == k)]) for k in range(pl.K)]
    y = oc.SparseConvFunction.apply(x, w, maps, pl.n_out)
    dy = cx.grid_operand(g, (pl.n_out, N), 2)
    y.backward(dy)
    got, _ = cx.gather_gemm(pl, x.detach(), w.detach().transpose(1, 2), flip=False)
    assert torch.equal(got, y.detach())
    # dgrad as lg_conv_gemm_tc runs it: the same pairs with in / out swapped, weights [K][N=Ck][Ck=N]
    swapped = cx.PairList(K=pl.K, n_slots=pl.n_in, n_out=pl.n_in, n_in=pl.n_out, k=pl.k[keep], slot=pl.inp[keep],
                          inp=rows[keep], out_row=None)
    dx, _ = cx.gather_gemm(swapped, dy, w.detach(), flip=False)
    assert torch.equal(dx, x.grad)
    dw, _ = cx.wgrad(pl, x.detach(), dy)
    assert torch.equal(dw, w.grad)


def _operands(case):
    g = torch.Generator().manual_seed(3)
    if isinstance(case, cx.GemmCase):
        pl = case.pairs(SM)
        n_in = pl.n_in
        return (cx.grid_operand(g, (n_in, case.Ck), case.ea), cx.grid_operand(g, (case.K, case.N, case.Ck), case.eb)), pl
    pl = case.pairs()
    return (cx.grid_operand(g, (pl.n_in, case.Cin), case.ea), cx.grid_operand(g, (pl.n_out, case.Cout), case.eb)), pl


@pytest.mark.parametrize("case", cx.GEMM_CASES + cx.WGRAD_CASES, ids=lambda c: c.name)
def test_grid_operands_are_exact_and_sums_stay_below_2_22(case):
    (a, b), pl = _operands(case)
    assert cx.round_trips(a) and cx.round_trips(b)
    if isinstance(case, cx.GemmCase):
        _, s_abs = cx.gather_gemm(pl, a, b, case.flip)
    else:
        _, s_abs = cx.wgrad(pl, a, b)
    assert cx.granules(s_abs, case.ea + case.eb) < cx.S_LIMIT


def test_gemm_grid_covers_every_branch_of_gemm2_shape():
    shapes = [c.shape(SM) for c in cx.GEMM_CASES]
    assert all(s is not None for s in shapes)
    assert {s["pc"] for s in shapes} == {1, 2, 3, 4}
    assert {s["T"] for s in shapes} == {1, 2, 3, 4}
    assert {s["n_split"] for s in shapes} == {1, 2}
    assert {s["n_split"] for s in shapes if s["rem16"]} == {1, 2}
    assert any(s["n_split"] == 2 and not c.flip for c, s in zip(cx.GEMM_CASES, shapes))  # n_split 2 in forward
    assert {s["sb"] for s in shapes} == {2, 3}
    assert any(s["fallback"] for s in shapes)
    assert any(s["n_panels"] > 1 for s in shapes)
    assert {c.Ck for c in cx.GEMM_CASES} >= {32, 64, 96, 128, 192, 256, 384, 512}
    assert {c.N for c in cx.GEMM_CASES} >= {16, 48, 96, 256, 288, 384, 512}
    assert all(s["T"] == c.T for c, s in zip(cx.GEMM_CASES, shapes) if c.T)  # rows sized for the T each case names
    k125 = [c for c in cx.GEMM_CASES if c.K == 125]
    assert {c.flip for c in k125} == {False, True}
    assert {(c.flip, c.scale, c.bias) for c in cx.GEMM_CASES} >= {(True, False, False), (False, True, False),
                                                                  (False, False, True)}


def test_wgrad_grid_covers_every_branch_of_wgrad2_shape():
    shapes = [(c, c.shape()) for c in cx.WGRAD_CASES]
    assert {c.Cout for c, _ in shapes} >= {32, 64, 128, 256}
    assert {c.Cin for c, _ in shapes} >= {32, 96, 160, 192, 384, 512}
    assert {s["K"] for _, s in shapes} >= {1, 8, 27, 64}
    assert {s["strided"] for _, s in shapes} == {False, True}
    assert {s["m_blocks"] for _, s in shapes} == {1, 2, 3, 4}
    assert any(c.Cin % 128 for c, s in shapes if s["m_blocks"] > 1)  # partly filled last channel block
    assert any(c.tiles == 1 for c, _ in shapes)
    assert any(1 < c.tiles < s["want"] for c, s in shapes)
    assert any(c.tiles % s["chunks"] for c, s in shapes)


def test_mirrors_reject_what_the_host_rejects():
    assert cx._gemm2_shape(100, 32, 400, SM) is None
    assert cx._gemm2_shape(100, 32, 336, SM) is None
    assert cx._gemm2_shape(100, 32, 48, SM, stats=True) is None


def test_minkunet34_shapes():
    shapes = cx.minkunet34_conv_shapes()
    assert len(shapes) == len(set(shapes))
    assert all(cin % 32 == 0 and cout % 32 == 0 for _, _, _, cin, cout in shapes)
    assert ("up", 16, 2, 256, 256) in shapes and ("same", 8, 3, 384, 256) in shapes
    assert ("identity", 1, 1, 128, 96) in shapes and ("down", 8, 2, 128, 128) in shapes
