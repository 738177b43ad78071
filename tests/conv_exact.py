"""Exact-operand checks of the convolution kernels: case grid, plan packer / validator and float64 oracle.

Operands are small integers times a power of two: x = i * 2^-a, w = j * 2^-b with |i|, |j| <= 8.  They are exact in
fp16 and bf16, every product is exact, and every partial sum is a multiple of the granule 2^-(a+b).  When
S = max over output elements of sum |x * w| / 2^-(a+b) stays below 2^22, no partial sum of any summation order has a
bit below one granule or above fp32's 24-bit significand, so an fp32 result must equal the float64 oracle bit for bit.
A missing, doubled or misrouted product then shows up in the element it belongs to, however large the output is.

This module has no GPU code: tests/test_conv_exact_host.py checks it on the CPU, tests/test_gpu_conv_exact.py runs the
kernels against it.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

TILE = 128
S_LIMIT = 2 ** 22
SM_COUNT_B200 = 148

# ------------------------------------------------------------------------------------------------ launch-shape mirrors
# Constants of lidog_b200/csrc/conv_tc2.cu (namespace lg::v2).
_K_SUB, _K_ROW_B, _K_IDX_SLOT_BYTES, _K_GEMM_IDX_SLOTS = 128 * 64, 64, TILE * 4, 16
_K_STG_BYTES = 4 * 32 * 36 * 4
_K_SCHED_SLOTS, _K_SCHED_WORDS, _K_PROD_WARPS = 4, 12, 4
_K_SMEM_BUDGET = 225 * 1024


def _ceil_div(a, b):
    return -(-a // b)


def _tail_bytes(sa, sb):
    # mirror of tail_bytes() in conv_tc2.cu
    ni = _K_GEMM_IDX_SLOTS
    return (ni * _K_IDX_SLOT_BYTES + _K_STG_BYTES + (2 * sa + 2 * sb + 2 * ni + 11 + 2 * _K_SCHED_SLOTS) * 8 + 16
            + 4 * _K_SCHED_WORDS * _K_SCHED_SLOTS + 1024)


def _gemm2_shape(n_tiles, Ck, N, sm_count, stats=False):
    """Line-for-line mirror of gemm2_shape() in lidog_b200/csrc/conv_tc2.cu (keep the two in step).
    -> dict of the launch shape, or None where the C function returns LG_ERR_UNSUPPORTED.  Used to label cases and to
    check that the grid reaches every branch; the kernels never see it."""
    n_split = (N + 255) // 256
    n_blk = N // n_split
    if n_blk % 16 != 0 or n_blk * n_split != N:
        return None
    if stats and n_blk % 32 != 0:
        return None
    if n_split > 4:
        return None
    n_chunks = Ck // 32
    n_panels = (n_chunks + 3) // 4
    while n_chunks % n_panels != 0:
        n_panels += 1
    pc = n_chunks // n_panels
    T = 256 // n_blk if 256 // n_blk < 4 else 4
    while T > 1 and _ceil_div(n_tiles, T) * n_split < 3 * sm_count:
        T -= 1
    fallback = False
    while True:
        stageA, stageB = pc * _K_SUB, pc * n_blk * _K_ROW_B
        sb = 3 if 3 * stageB + 4 * stageA + _tail_bytes(4, 3) <= _K_SMEM_BUDGET else 2
        sa = 12
        while sa > 2 and sa * stageA + sb * stageB + _tail_bytes(sa, sb) > _K_SMEM_BUDGET:
            sa -= 1
        if sb == 3 and sa < 12 and stageB <= stageA:
            sa2 = 12
            while sa2 > 2 and sa2 * stageA + 2 * stageB + _tail_bytes(sa2, 2) > _K_SMEM_BUDGET:
                sa2 -= 1
            if sa2 > sa:
                sa, sb = sa2, 2
        if sa >= _K_PROD_WARPS or pc == 1:
            break
        pc -= 1  # deeper ring with smaller panels
        while n_chunks % pc != 0:
            pc -= 1
        n_panels = n_chunks // pc
        fallback = True
    T = T if T < sa else sa
    smem = sa * stageA + sb * stageB + _tail_bytes(sa, sb)
    if smem > _K_SMEM_BUDGET:
        return None
    return dict(n_split=n_split, n_blk=n_blk, T=T, pc=pc, n_panels=n_panels, sa=sa, sb=sb,
                np=min(sa, _K_PROD_WARPS), n_super=_ceil_div(n_tiles, T), rem16=n_blk % 32 == 16, fallback=fallback)


def _wgrad2_shape(K, n_tiles, Cin, Cout):
    """Line-for-line mirror of wgrad2_shape() and the group choice of launch_wgrad_tc2() in
    lidog_b200/csrc/conv_tc2.cu (keep the two in step).  -> dict of the launch shape."""
    gmax = 512 // Cout
    if gmax > 8:
        gmax = 8
    if gmax > K:
        gmax = K
    n_groups = (K + gmax - 1) // gmax
    G = (K + n_groups - 1) // n_groups
    m_blocks = (Cin + 127) // 128
    per = n_groups * m_blocks
    hi, lo = 592 // per, _ceil_div(148, per)
    want = n_tiles // 32
    want = max(min(max(want, lo), hi), 1)
    chunks = max(min(n_tiles, want), 1)
    tpc = _ceil_div(max(n_tiles, 1), chunks)
    chunks_launched = _ceil_div(max(n_tiles, 1), tpc)
    return dict(G=G, n_groups=n_groups, strided=n_groups >= 5, m_blocks=m_blocks, K=K, want=want,
                chunks=chunks_launched, tiles_per_chunk=tpc)


def gemm_label(sh):
    return f"pc={sh['pc']} T={sh['T']} n_split={sh['n_split']}" + (" rem16" if sh["rem16"] else "") + \
        f" sb={sh['sb']}" + (" fallback" if sh["fallback"] else "")


def wgrad_label(sh, n_tiles):
    chunking = "one-tile" if n_tiles == 1 else ("few-tiles" if n_tiles < sh["want"] else "")
    if n_tiles % sh["chunks"]:
        chunking += " ragged-chunks"
    chunking = chunking.strip()
    return (f"n_groups={sh['n_groups']} {'strided' if sh['strided'] else 'contiguous'} m_blocks={sh['m_blocks']} "
            f"K={sh['K']} chunks={sh['chunks']} {chunking}").strip()


# ------------------------------------------------------------------------------------------------ operands
def grid_operand(gen: torch.Generator, shape, exp: int, imax: int = 8, p_zero: float = 0.25) -> torch.Tensor:
    """float64 values i * 2^-exp, i uniform in [-imax, imax], a fraction p_zero of them exactly zero."""
    i = torch.randint(-imax, imax + 1, shape, generator=gen, dtype=torch.int64)
    i[torch.rand(shape, generator=gen, dtype=torch.float64) < p_zero] = 0
    return i.double() * 2.0 ** -exp


def round_trips(t: torch.Tensor) -> bool:
    """t (float64) survives float64 -> fp16 / bf16 / fp32 -> float64 unchanged."""
    return all(torch.equal(t.to(dt).double(), t) for dt in (torch.float16, torch.bfloat16, torch.float32))


# ------------------------------------------------------------------------------------------------ hand-built plans
@dataclass
class PairList:
    """The convolution as a list of (offset k, slot s, input row i) products; slot s feeds result row out_row[s]
    (natural order: s itself when s < n_out), padding slots (-1 / >= n_out) feed nothing."""
    K: int
    n_slots: int
    n_out: int
    n_in: int
    k: np.ndarray
    slot: np.ndarray
    inp: np.ndarray
    out_row: np.ndarray | None  # int64 [n_slots] or None (natural order)
    extra_mask: np.ndarray = field(default=None)  # bool [n_tiles, K]: offsets a tile announces without any pair
    k_stride0: bool = False  # one nbr row shared by every offset (each tile then has a single offset)

    @property
    def n_tiles(self):
        return self.n_slots // TILE

    def result_rows(self) -> np.ndarray:
        """Result row of each pair's slot (-1 = padding)."""
        if self.out_row is None:
            r = self.slot.copy()
            r[r >= self.n_out] = -1
            return r
        return self.out_row[self.slot]


def make_pairs(rng: np.random.Generator, K, n_tiles, n_out=None, n_in=None, order="natural", masks="random",
               density=0.6, k_stride0=False, edges=True) -> PairList:
    """Random pair list of a plan of n_tiles tiles.

    order: "natural" (slot s = row s) or "perm" (out_row a random permutation, padding slots scattered).
    masks: "random" (each tile a random offset subset, some tiles empty), "alt_empty" (every other tile empty),
           "hi_lo" (tiles using only offsets >= 32, only offsets < 32, or both, in turn), "one" (one offset per tile).
    edges: tile 0 gathers one input row in all 128 slots of its first offset, tile 1 announces an offset whose slots
           are all -1, tile 2 is empty.
    """
    n_slots = n_tiles * TILE
    n_out = n_slots if n_out is None else n_out
    n_in = n_out if n_in is None else n_in
    tiles = np.arange(n_tiles)
    if masks == "random":
        m = rng.random((n_tiles, K)) < 0.5
        m[rng.random(n_tiles) < 0.1] = False
    elif masks == "alt_empty":
        m = rng.random((n_tiles, K)) < 0.5
        m[:, 0] |= True
        m[1::2] = False
    elif masks == "hi_lo":
        assert K > 32
        m = rng.random((n_tiles, K)) < 0.25
        m[tiles % 3 == 0, :32] = False
        m[tiles % 3 == 1, 32:] = False
        m[tiles % 3 == 0, 32 + (tiles[tiles % 3 == 0] % (K - 32))] = True
        m[tiles % 3 == 1, tiles[tiles % 3 == 1] % 32] = True
    elif masks == "one":
        m = np.zeros((n_tiles, K), bool)
        m[tiles, rng.integers(0, K, n_tiles)] = True
    else:
        raise ValueError(masks)
    extra = np.zeros((n_tiles, K), bool)
    slot_tile = np.arange(n_slots) // TILE
    take = m[slot_tile].T & (rng.random((K, n_slots)) < density)  # [K, n_slots]
    src = rng.integers(0, n_in, (K, n_slots))
    if edges and n_tiles >= 3:
        # tile 0: every slot of its first offset gathers the same input row
        k0 = int(np.flatnonzero(m[0])[0]) if m[0].any() else 0
        take[k0, :TILE] = True
        src[k0, :TILE] = rng.integers(0, n_in)
        # tile 1: one offset is announced in the mask, but all of its slots are -1
        k1 = int(np.flatnonzero(m[1])[0]) if m[1].any() else 0
        take[k1, TILE:2 * TILE] = False
        extra[1, k1] = True
        # tile 2: no offset at all
        take[:, 2 * TILE:3 * TILE] = False
    ks, slots = np.nonzero(take)
    inp = src[ks, slots]
    out_row = None
    if order == "perm":
        out_row = rng.permutation(n_slots).astype(np.int64)
        out_row[out_row >= n_out] = -1
    elif order != "natural":
        raise ValueError(order)
    return PairList(K, n_slots, n_out, n_in, ks.astype(np.int64), slots.astype(np.int64), inp.astype(np.int64),
                    out_row, extra, k_stride0)


def pack_plan(pl: PairList):
    """Pair list -> the (nbr, out_row, tile_mask) arrays of an lgConvPlan (int32 / uint32-as-int32 numpy arrays)."""
    words = (pl.K + 31) // 32
    if pl.k_stride0:
        assert np.unique(pl.slot).size == pl.slot.size, "k_stride = 0 takes one offset per slot"
        nbr = np.full(pl.n_slots, -1, np.int64)
        nbr[pl.slot] = pl.inp
    else:
        nbr = np.full((pl.K, pl.n_slots), -1, np.int64)
        nbr[pl.k, pl.slot] = pl.inp
    bits = np.zeros((pl.n_tiles, pl.K), bool)
    bits[pl.slot // TILE, pl.k] = True
    if pl.extra_mask is not None:
        bits |= pl.extra_mask
    mask = np.zeros((pl.n_tiles, words), np.uint32)
    for k in range(pl.K):
        mask[:, k // 32] |= bits[:, k].astype(np.uint32) << np.uint32(k % 32)
    out_row = None if pl.out_row is None else pl.out_row.astype(np.int32)
    return nbr.astype(np.int32), out_row, mask.view(np.int32), (0 if pl.k_stride0 else pl.n_slots)


def validate_plan(nbr, k_stride, out_row, tile_mask, K, n_slots, n_out, n_in):
    """Raise AssertionError unless the plan is safe to hand to a kernel: every gather and every store in range."""
    assert n_slots > 0 and n_slots % TILE == 0, "n_slots must be a positive multiple of 128"
    words = (K + 31) // 32
    assert tile_mask.shape == (n_slots // TILE, words), tile_mask.shape
    assert k_stride in (0, n_slots)
    assert nbr.shape == ((n_slots,) if k_stride == 0 else (K, n_slots)), nbr.shape
    assert nbr.min() >= -1 and nbr.max() < n_in, "nbr out of [-1, n_in)"
    if out_row is not None:
        assert out_row.shape == (n_slots,)
        assert out_row.min() >= -1 and out_row.max() < n_out, "out_row out of [-1, n_out)"
        rows = out_row[out_row >= 0]
        assert np.unique(rows).size == rows.size, "a result row written by two slots"
    m = tile_mask.view(np.uint32)
    if K % 32:
        assert not (m[:, -1] >> np.uint32(K % 32)).any(), "mask bit >= K"


def plan_of_pairs(pl: PairList, **override):
    """Packed, validated plan arrays of a pair list (dict of numpy arrays and sizes)."""
    nbr, out_row, mask, k_stride = pack_plan(pl)
    p = dict(nbr=nbr, k_stride=k_stride, out_row=out_row, tile_mask=mask, K=pl.K, n_slots=pl.n_slots,
             n_out=pl.n_out, n_in=pl.n_in)
    p.update(override)
    validate_plan(**p)
    return p


# ------------------------------------------------------------------------------------------------ float64 oracle
def gather_gemm(pl: PairList, A: torch.Tensor, B: torch.Tensor, flip: bool):
    """Y[row(s)] = sum over pairs (k, s, i) of A[i] @ B[wk]^T, wk = K-1-k when flip; B is [K][N][Ck] (the layout of
    lg_conv_gemm_tc).  -> (Y float64 [n_out, N], S = max_row,col sum |A| |B| in units of the smallest granule)."""
    rows = torch.from_numpy(pl.result_rows())
    keep = rows >= 0
    k, i, r = torch.from_numpy(pl.k)[keep], torch.from_numpy(pl.inp)[keep], rows[keep]
    N = B.shape[1]
    Y = torch.zeros(pl.n_out, N, dtype=torch.float64)
    Yabs = torch.zeros(pl.n_out, N, dtype=torch.float64)
    for kk in torch.unique(k).tolist():
        sel = k == kk
        wk = pl.K - 1 - kk if flip else kk
        a = A.index_select(0, i[sel])
        Y.index_add_(0, r[sel], a @ B[wk].t())
        Yabs.index_add_(0, r[sel], a.abs() @ B[wk].abs().t())
    return Y, Yabs


def wgrad(pl: PairList, X: torch.Tensor, dY: torch.Tensor):
    """dW[k] = sum over pairs (k, s, i) with a result row of X[i]^T dY[row(s)].  -> (dW [K][Cin][Cout], |dW| sum)."""
    rows = torch.from_numpy(pl.result_rows())
    keep = rows >= 0
    k, i, r = torch.from_numpy(pl.k)[keep], torch.from_numpy(pl.inp)[keep], rows[keep]
    dW = torch.zeros(pl.K, X.shape[1], dY.shape[1], dtype=torch.float64)
    dWabs = torch.zeros_like(dW)
    for kk in torch.unique(k).tolist():
        sel = k == kk
        a, b = X.index_select(0, i[sel]), dY.index_select(0, r[sel])
        dW[kk] = a.t() @ b
        dWabs[kk] = a.abs().t() @ b.abs()
    return dW, dWabs


def granules(abs_sum: torch.Tensor, exp: int) -> float:
    """S: the largest sum of |products| in units of the granule 2^-exp."""
    return float(abs_sum.max()) * 2.0 ** exp if abs_sum.numel() else 0.0


# ------------------------------------------------------------------------------------------------ case grid
@dataclass(frozen=True)
class GemmCase:
    """A gather-GEMM launch on a hand-built plan.  T is the super-tile depth the row count is sized for (n_tiles is
    derived from the SM count); tiles is the tile count when T is None."""
    name: str
    Ck: int
    N: int
    K: int
    T: int | None = None
    tiles: int = 24
    order: str = "natural"
    masks: str = "random"
    flip: bool = False
    scale: bool = False
    bias: bool = False
    n_in: int | None = None
    n_out_minus: int = 0  # n_out = n_slots - n_out_minus (natural order: a ragged last tile)
    k_stride0: bool = False
    ea: int = 3  # x = i * 2^-ea
    eb: int = 6  # w = j * 2^-eb

    def n_tiles(self, sm_count):
        if self.T is None:
            return self.tiles
        n_split = (self.N + 255) // 256
        per = _ceil_div(3 * sm_count, n_split)  # super-tiles that keep T from being lowered
        return per * self.T - (1 if self.T > 1 else 0)  # and a partial last super-tile

    def shape(self, sm_count):
        return _gemm2_shape(self.n_tiles(sm_count), self.Ck, self.N, sm_count)

    def pairs(self, sm_count):
        rng = np.random.default_rng(_seed(self.name))
        n_tiles = self.n_tiles(sm_count)
        n_out = n_tiles * TILE - self.n_out_minus
        return make_pairs(rng, self.K, n_tiles, n_out=n_out, n_in=self.n_in, order=self.order, masks=self.masks,
                          k_stride0=self.k_stride0, density=0.6 if self.K > 1 else 0.9)


def _seed(name: str) -> int:
    return int.from_bytes(name.encode()[:8].ljust(8, b"\0"), "little") % (2 ** 32)


GEMM_CASES = [
    # super-tile depth T = 4 / 3 / 2 (two accumulator sets, several waves of the dynamic hand-out)
    GemmCase("T4_rem16", 32, 16, 1, T=4, bias=True),
    GemmCase("T3_rem16_perm", 64, 48, 1, T=3, order="perm", scale=True),
    GemmCase("T2_alt_empty_dgrad", 128, 96, 8, T=2, masks="alt_empty", flip=True),
    GemmCase("T2_pc1", 32, 128, 2, T=2, order="perm", bias=True),
    # operand widths: pc = 1..4, several panels; column blocks: n_split 1 / 2, the 16-column remainder
    GemmCase("ck64_n64", 64, 64, 8, scale=True),
    GemmCase("ck96_n96_pc3", 96, 96, 8, order="perm"),
    GemmCase("ck192_n288_split2_rem16", 192, 288, 8, flip=True, scale=True),
    GemmCase("ck256_n256_fallback", 256, 256, 8, bias=True),
    GemmCase("ck384_n384_split2", 384, 384, 8, order="perm", flip=True),
    GemmCase("ck512_n512_split2", 512, 512, 8, scale=True, bias=True),
    GemmCase("ck128_n16_rem16", 128, 16, 8, order="perm", flip=True),
    GemmCase("ck32_n48_rem16", 32, 48, 27, bias=True),
    GemmCase("ck512_n96", 512, 96, 8, flip=True),
    # plan edges
    GemmCase("n_in_1", 64, 32, 8, n_in=1),
    GemmCase("last_tile_one_row", 32, 64, 8, tiles=5, n_out_minus=127, bias=True),
    GemmCase("k_stride0_one_offset", 96, 128, 8, masks="one", k_stride0=True, order="perm"),
    GemmCase("single_tile", 32, 32, 27, tiles=1, n_out_minus=100),
    # kernel volume 125: four mask words, tiles with offsets only >= 32, only < 32, or both
    GemmCase("K125_fwd", 32, 64, 125, masks="hi_lo", bias=True),
    GemmCase("K125_dgrad", 64, 32, 125, masks="hi_lo", flip=True, scale=True, order="perm"),
]


@dataclass(frozen=True)
class WgradCase:
    name: str
    Cin: int
    Cout: int
    K: int
    tiles: int
    order: str = "natural"
    masks: str = "random"
    n_out_minus: int = 0
    k_stride0: bool = False
    ea: int = 3
    eb: int = 5

    def shape(self):
        return _wgrad2_shape(self.K, self.tiles, self.Cin, self.Cout)

    def pairs(self):
        rng = np.random.default_rng(_seed("w" + self.name))
        n_out = self.tiles * TILE - self.n_out_minus
        return make_pairs(rng, self.K, self.tiles, n_out=n_out, order=self.order, masks=self.masks,
                          k_stride0=self.k_stride0)


WGRAD_CASES = [
    WgradCase("one_tile", 32, 32, 27, 1, n_out_minus=60),
    WgradCase("few_tiles", 96, 64, 8, 5, order="perm"),
    WgradCase("mb2_partial_K64", 160, 128, 64, 37),
    WgradCase("mb2_strided_K27", 192, 256, 27, 20, order="perm"),
    WgradCase("mb3_K1", 384, 32, 1, 64),
    WgradCase("mb4_K8", 512, 64, 8, 40, order="perm", n_out_minus=5),
    WgradCase("K64_cout32_strided", 32, 32, 64, 11),
    WgradCase("K64_cout256", 96, 256, 64, 9, order="perm"),
    WgradCase("K27_contiguous", 160, 64, 27, 33),
    WgradCase("K8_cout128", 192, 128, 8, 64, masks="alt_empty"),
    WgradCase("k_stride0", 64, 64, 8, 16, masks="one", k_stride0=True, order="perm"),
]


# ------------------------------------------------------------------------------------------------ MinkUNet34 layers
def minkunet34_conv_shapes():
    """Distinct (kind, tensor stride in, kernel size, Cin, Cout) of the tensor-core convolutions of MinkUNet34BEV,
    derived from lidog_b200/lidog/model.py as its constructor builds them: stride-2 encoder convolutions, residual
    stages (3x3x3 convolutions and 1x1 downsample projections where the width changes), transposed decoder
    convolutions whose stage input is the concatenation with the encoder skip.  The 5x5x5 stem (Cin = 1) and the
    class head (Cout = classes) are not multiples of 32 and run on the fp32 SIMT kernels."""
    from lidog_b200.lidog.model import INIT_DIM, LAYERS34, PLANES
    shapes = []
    inplanes = INIT_DIM

    def stage(planes, ts, n):
        nonlocal inplanes
        if inplanes != planes:
            shapes.append(("identity", ts, 1, inplanes, planes))
        shapes.append(("same", ts, 3, inplanes, planes))
        shapes.append(("same", ts, 3, planes, planes))
        inplanes = planes
        assert n >= 1

    for i, ts in enumerate((1, 2, 4, 8)):
        shapes.append(("down", ts, 2, inplanes, inplanes))
        stage(PLANES[i], 2 * ts, LAYERS34[i])
    skips = (PLANES[2], PLANES[1], PLANES[0], INIT_DIM)
    for j, ts in enumerate((16, 8, 4, 2)):
        i = 4 + j
        shapes.append(("up", ts, 2, inplanes, PLANES[i]))
        inplanes = PLANES[i] + skips[j]
        stage(PLANES[i], ts // 2, LAYERS34[i])
    out = []
    for s in shapes:
        if s not in out:
            out.append(s)
    return out
