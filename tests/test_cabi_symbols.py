"""CPU: the C-ABI library builds, loads and exports every symbol include/lidog_b200.h declares
(no compute without a GPU), and the host layer mirrors the MinkowskiEngine surface."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    from lidog_b200 import build
    return build.build()


def _declared():
    src = open(os.path.join(ROOT, "include", "lidog_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lg_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(libpath):
    names = _declared()
    assert len(names) >= 20
    lib = ctypes.CDLL(libpath)
    for n in names:
        assert hasattr(lib, n), n
    from lidog_b200 import cabi
    assert sorted(cabi.SIGNATURES) == names  # the binding covers the header exactly


def test_host_only_entry_points(libpath):
    from lidog_b200 import cabi
    L = cabi.lib()
    assert L.lg_version() >= 100
    assert L.lg_hash_capacity(1000) == 2048 and L.lg_hash_capacity(0) == 1024
    assert L.lg_hash_bytes(2048) == 2048 * 16
    assert L.lg_coords_unique_workspace(1000) > 8000
    # argument validation happens before any CUDA call
    assert L.lg_quantize_points(None, None, -1, 0.05, 0.05, 0.05, None, None) == -1
    assert b"lg_quantize_points" in L.lg_last_error_string()
    assert L.lg_quantize_points_f64(None, None, 0, 0.05, 0.05, 0.05, None, None) == 0   # empty cloud: nothing to do
    assert L.lg_quantize_points_f64(None, None, 5, 0.05, 0.0, 0.05, None, None) == -1   # doubles arrive as doubles
    assert L.lg_quantize_points_f64(None, None, 5, 0.05, 0.05, 0.05, None, None) == -1  # null pointers
    assert b"lg_quantize_points_f64: null pointer" in L.lg_last_error_string()


def test_sass_contains_blackwell_tensor_and_tma_instructions(libpath):
    import subprocess
    sass = subprocess.run(["cuobjdump", "-sass", libpath], capture_output=True, text=True).stdout
    # what the LIVE path emits (B200_PROFILING.md): tcgen05.mma, tcgen05.ld, tiled TMA (weight panels), bulk copies
    # (row-id ring), cp.async (row gathers), mbarrier
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG.2D", "UBLKCP", "LDGSTS", "SYNCS"):
        assert mnemonic in sass, mnemonic
    # the first-generation gather4 kernels are not in the product library any more
    assert "GATHER4" not in sass


def test_minkowski_engine_surface_matches_reference_usage():
    import MinkowskiEngine as ME
    for name in ("SparseTensor", "MinkowskiConvolution", "MinkowskiConvolutionTranspose", "MinkowskiBatchNorm",
                 "MinkowskiSyncBatchNorm", "MinkowskiReLU", "MinkowskiDropout", "cat"):
        assert hasattr(ME, name), name
    for name in ("sparse_quantize", "SparseCollation", "kaiming_normal_", "batched_coordinates"):
        assert hasattr(ME.utils, name), name
    from MinkowskiEngine.modules.resnet_block import BasicBlock, Bottleneck
    assert BasicBlock.expansion == 1 and Bottleneck.expansion == 4
    conv = ME.MinkowskiConvolution(32, 64, kernel_size=3, dimension=3)
    assert tuple(conv.kernel.shape) == (27, 32, 64) and conv.bias is None
    assert tuple(ME.MinkowskiConvolution(96, 7, kernel_size=1, bias=True, dimension=3).kernel.shape) == (96, 7)
    assert tuple(ME.MinkowskiConvolutionTranspose(8, 4, kernel_size=2, stride=2, dimension=3).kernel.shape) == (8, 8, 4)
    assert not isinstance(ME.MinkowskiConvolutionTranspose(8, 4, kernel_size=2, stride=2, dimension=3),
                          ME.MinkowskiConvolution)  # kaiming init must skip transposed convs (minkunet_bev.py:403)
    bn = ME.MinkowskiBatchNorm(32)
    assert isinstance(bn.bn, torch.nn.BatchNorm1d)
    sync = ME.MinkowskiSyncBatchNorm.convert_sync_batchnorm(torch.nn.Sequential(conv, ME.MinkowskiBatchNorm(64)))
    assert isinstance(sync[1], ME.MinkowskiSyncBatchNorm) and isinstance(sync[1].bn, torch.nn.SyncBatchNorm)
    t = torch.empty(27, 16, 32)
    ME.utils.kaiming_normal_(t, mode="fan_out", nonlinearity="relu")
    assert abs(float(t.std()) - (2.0 / (32 * 27)) ** 0.5) < 0.01
    coords, feats, labels = ME.utils.SparseCollation(dtype=torch.float32)(
        [(torch.zeros(2, 3, dtype=torch.int32), torch.ones(2, 1), torch.zeros(2)),
         (torch.ones(3, 3, dtype=torch.int32), torch.ones(3, 1), torch.ones(3))])
    assert coords.dtype == torch.float32 and coords[:, 0].tolist() == [0, 0, 1, 1, 1] and feats.shape == (5, 1)


def test_no_cpu_fallback():
    import MinkowskiEngine as ME
    with pytest.raises(RuntimeError, match="no CPU path"):
        ME.SparseTensor(coordinates=torch.zeros(4, 4, dtype=torch.int32), features=torch.ones(4, 1))


def test_model_state_dict_matches_reference_names():
    """Parameter names/shapes of the table-driven model equal the reference class's (checked against
    the unchanged reference file when a checkout of it is at oracle/_ref/, else against the expected counts)."""
    from lidog_b200.lidog.model import MinkUNet34BEV
    import MinkowskiEngine as ME
    from tests import refharness as rh
    m = MinkUNet34BEV(1, 7)
    sd = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert len(sd) == 388 and sum(p.numel() for p in m.parameters()) == 38_660_622
    assert sd["conv0p1s1.kernel"] == (125, 1, 32) and sd["final.kernel"] == (96, 7) and sd["final.bias"] == (1, 7)
    assert sd["block5.0.downsample.0.kernel"] == (384, 256) and sd["convtr4p16s2.kernel"] == (8, 256, 256)
    assert "encoders2d.block8.down1.maxpool_conv.0.double_conv.0.weight" in sd
    if rh.reference_available():
        import sys
        sys.path.insert(0, rh.REF)
        try:
            import utils.models.minkunet_bev as ref  # the UNCHANGED reference file on the drop-in package
            r = ref.MinkUNet34BEV(1, 7, 3)
            assert {k: tuple(v.shape) for k, v in r.state_dict().items()} == sd
        finally:
            sys.path.remove(rh.REF)


def test_wgrad_workspace_covers_the_chunk_rule(libpath):
    """`lg_conv_wgrad_tc_workspace` is host-only and must cover the partial-dW buffers of `k_wgrad2`:
    chunks x K x Cin x Cout floats, chunks = tiles / 32 clamped to [one wave of 148 CTAs, four waves] over the
    (offset group x 128-channel block) CTAs (csrc/conv_tc2.cu, from the CTA sweep in profiles/r01_s4_sweep_a.txt).
    (The entry point returns the maximum over the kernel generations, so this is a lower bound.)"""
    import math
    import os
    from lidog_b200 import cabi
    os.environ.pop("LIDOG_WG_CTAS", None)
    L = cabi.lib()

    def workspace(n_tiles, K, cin, cout):
        plan = cabi.ConvPlan(None, 128 * n_tiles, None, None, K, (K + 31) // 32, 128 * n_tiles, 128 * n_tiles,
                             128 * n_tiles)
        return L.lg_conv_wgrad_tc_workspace(plan, cin, cout)

    def rule(n_tiles, K, cin, cout):
        gmax = min(512 // cout, 8, K)
        per = math.ceil(K / gmax) * math.ceil(cin / 128)
        want = min(max(n_tiles // 32, math.ceil(148 / per)), max(592 // per, 1))
        c = max(1, min(n_tiles, want))
        return math.ceil(n_tiles / math.ceil(n_tiles / c))

    for shape in [(5065, 27, 96, 96), (2463, 27, 96, 96), (964, 27, 128, 128), (353, 27, 256, 256),
                  (129, 27, 256, 256), (353, 27, 128, 128), (964, 27, 64, 64), (5065, 8, 32, 32), (5065, 1, 128, 96),
                  (3, 27, 384, 256)]:
        n_tiles, K, cin, cout = shape
        assert workspace(*shape) >= rule(*shape) * K * cin * cout * 4 + 256, shape
    assert rule(129, 27, 256, 256) == 6 and rule(5065, 27, 96, 96) == 98  # the two ends of the sweep
    assert workspace(0, 27, 96, 96) > 0 and L.lg_conv_wgrad_tc_workspace(None, 96, 96) == 0
