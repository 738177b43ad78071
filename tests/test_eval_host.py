"""CPU: the evaluation path's host logic -- IoU from the confusion matrix in both reference conventions, argument
validation of lg_conv_layer_infer / lg_confusion_matrix before any CUDA call, and the conditions under which a
convolution forward takes the inference epilogue."""
import ctypes

import numpy as np
import pytest
import torch

from lidog_b200.lidog.evaluate import iou_from_confusion

LG_ERR_INVALID, LG_ERR_UNSUPPORTED = -1, -4


@pytest.fixture(scope="module")
def L():
    from lidog_b200 import build, cabi
    build.build()
    return cabi.lib()


def _confusion(target, pred, C):
    """(C + 1) x C counts, row C = targets outside [0, C) -- what lg_confusion_matrix accumulates."""
    row = np.where((target >= 0) & (target < C), target, C)
    conf = np.zeros((C + 1, C), dtype=np.int64)
    np.add.at(conf, (row, pred), 1)
    return conf


def _labels(rng, n, C, out_of_range):
    t = rng.integers(0, C, n)
    t[rng.random(n) < 0.15] = -1                       # ignore label
    if out_of_range:
        t[rng.random(n) < 0.05] = C + rng.integers(0, 3)  # labels the head does not predict
    t[t == 2] = 0                                       # class 2 never a target
    p = rng.integers(0, C, n)
    p[p == 3] = 1                                       # class 3 never predicted
    if C > 5:
        p[p == 5] = 4
        t[t == 5] = 4                                   # class 5 absent from both: IoU 0
    return t, p


@pytest.mark.parametrize("C", [7, 19])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_iou_matches_sklearn_jaccard_score(C, seed):
    from sklearn.metrics import jaccard_score
    rng = np.random.default_rng(seed)
    t, p = _labels(rng, 5000, C, out_of_range=True)
    got = iou_from_confusion(_confusion(t, p, C), ignore_rows=False)
    want = jaccard_score(t, p, labels=list(range(C)), average=None, zero_division=0)
    assert np.array_equal(got, want)
    # the score is symmetric in its two arguments over the classes it reports
    assert np.array_equal(got, jaccard_score(p, t, labels=list(range(C)), average=None, zero_division=0))


@pytest.mark.parametrize("C", [7, 19])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_iou_ignoring_rows_matches_torchmetrics_jaccard(C, seed):
    from tests.refharness import _JaccardIndex
    rng = np.random.default_rng(seed)
    t, p = _labels(rng, 5000, C, out_of_range=False)
    got = iou_from_confusion(_confusion(t, p, C), ignore_rows=True)
    want = _JaccardIndex(C, ignore_index=-1)(torch.from_numpy(p), torch.from_numpy(t)).numpy()
    assert want.dtype == np.float32
    assert np.array_equal(got.astype(np.float32), want)
    # every target outside [0, C) lands in row C, so all of them are dropped in this convention
    t2, p2 = _labels(rng, 5000, C, out_of_range=True)
    t2m = np.where((t2 >= 0) & (t2 < C), t2, -1)
    want2 = _JaccardIndex(C, ignore_index=-1)(torch.from_numpy(p2), torch.from_numpy(t2m)).numpy()
    assert np.array_equal(iou_from_confusion(_confusion(t2, p2, C), ignore_rows=True).astype(np.float32), want2)


def test_iou_of_an_empty_matrix_is_zero():
    assert np.array_equal(iou_from_confusion(np.zeros((8, 7), np.int64), ignore_rows=False), np.zeros(7))
    assert np.array_equal(iou_from_confusion(np.zeros((8, 7), np.int64), ignore_rows=True), np.zeros(7))


def _plan(cabi, K=27, n_tiles=3):
    fake = 0x10000  # never dereferenced: validation happens before any CUDA call
    n = 128 * n_tiles
    return cabi.ConvPlan(fake, n, None, fake, K, (K + 31) // 32, n, n, n)


def test_conv_layer_infer_validates_before_cuda(L):
    from lidog_b200 import cabi
    p = ctypes.byref(_plan(cabi))
    a = 0x20000  # 16-byte aligned stand-in pointers

    def call(plan=p, X16=a, Cin=64, W=None, Cout=64, w16=None, w16t=a, prep=0, fmt=cabi.FMT_FP16, st=a, res=None,
             relu=1, Y=a, Y16=a):
        return L.lg_conv_layer_infer(plan, X16, Cin, W, Cout, w16, w16t, prep, fmt, st, res, relu, Y, Y16, None)

    for kw in (dict(X16=None), dict(w16t=None), dict(Y=None), dict(st=None), dict(prep=1), dict(prep=1, W=a),
               dict(plan=None)):
        assert call(**kw) == LG_ERR_INVALID, kw
        assert b"lg_conv_layer_infer" in L.lg_last_error_string()
    assert call(res=a + 4) == LG_ERR_INVALID and b"aligned" in L.lg_last_error_string()
    assert call(Y16=a + 2) == LG_ERR_INVALID
    assert call(fmt=7) == LG_ERR_INVALID
    # column blocks of k_gemm2 that are not multiples of 32: a 16-column remainder path is not built
    for cout in (48, 80, 288):
        assert call(Cout=cout) == LG_ERR_UNSUPPORTED, cout
        assert b"multiples of 32" in L.lg_last_error_string()
    assert call(Cin=48) == LG_ERR_UNSUPPORTED  # operand chunks of 32 channels, as lg_conv_layer_forward


def test_confusion_matrix_validates_before_cuda(L):
    a = 0x20000
    assert L.lg_confusion_matrix(None, 0, 7, None, None, None) == 0  # nothing to do
    assert L.lg_confusion_matrix(a, 10, 0, a, a, None) == LG_ERR_INVALID
    assert L.lg_confusion_matrix(a, 10, 33, a, a, None) == LG_ERR_INVALID
    assert L.lg_confusion_matrix(a, -1, 7, a, a, None) == LG_ERR_INVALID
    for args in ((None, a, a), (a, None, a), (a, a, None)):
        assert L.lg_confusion_matrix(args[0], 10, 7, args[1], args[2], None) == LG_ERR_INVALID
        assert b"lg_confusion_matrix: null pointer" in L.lg_last_error_string()
    for args in ((a, a, a + 4), (a, a + 4, a), (a + 2, a, a)):
        assert L.lg_confusion_matrix(args[0], 10, 7, args[1], args[2], None) == LG_ERR_INVALID
        assert b"aligned" in L.lg_last_error_string()


def test_evaluator_rejects_host_tensors():
    from lidog_b200.lidog.evaluate import LidogEvaluator
    ev = LidogEvaluator(None, 7)
    with pytest.raises(ValueError, match="CUDA"):
        ev.add(torch.zeros(4, 7), torch.zeros(4, dtype=torch.int64))


def test_deferred_conv_only_in_eval_without_grad():
    from lidog_b200.me import conv
    ok = dict(training=False, grad_enabled=False, has_bias=False, cin=96, cout=96, is_cuda=True, n_out=1000)
    assert conv.infer_fast_path(**ok)
    for change in (dict(training=True), dict(grad_enabled=True), dict(training=True, grad_enabled=True),
                   dict(has_bias=True), dict(cin=1), dict(cout=7), dict(cout=288), dict(is_cuda=False),
                   dict(n_out=0)):
        assert not conv.infer_fast_path(**{**ok, **change}), change
    for cin, cout in ((32, 32), (64, 64), (128, 96), (384, 256), (256, 128)):
        assert conv.infer_fast_path(**{**ok, "cin": cin, "cout": cout})
    for key, off in (("tc", "off"), ("layer_calls", 0)):
        saved = conv.CONFIG[key]
        conv.CONFIG[key] = off
        try:
            assert not conv.infer_fast_path(**ok), key
        finally:
            conv.CONFIG[key] = saved
    conv.PROFILE["enabled"] = True
    try:
        assert not conv.infer_fast_path(**ok)
    finally:
        conv.PROFILE["enabled"] = False


def test_eval_bn_coefficients_follow_torch_eval_batch_norm():
    from lidog_b200.me.norm import MinkowskiBatchNorm, eval_bn_stats
    torch.manual_seed(0)
    m = MinkowskiBatchNorm(64)
    with torch.no_grad():
        m.bn.weight.uniform_(0.5, 2.0)
        m.bn.bias.uniform_(-1, 1)
        m.bn.running_mean.uniform_(-1, 1)
        m.bn.running_var.uniform_(0.1, 3.0)
    m.eval()
    st = eval_bn_stats(m.bn)
    assert st.dtype == torch.float32 and st.shape == (256,)
    x = torch.randn(500, 64, dtype=torch.float64)
    want = m.bn.double()(x)
    got = x * st[128:192].double() + st[192:].double()
    assert torch.allclose(got, want, rtol=1e-6, atol=1e-6)
    m.bn.float()
    # cached until a parameter / buffer changes or the module goes back to training mode
    s1 = m._eval_stats()
    assert m._eval_stats() is s1
    with torch.no_grad():
        m.bn.running_var.mul_(2.0)
    s2 = m._eval_stats()
    assert s2 is not s1 and not torch.equal(s1, s2)
    m.eval()  # (LidogEvaluator switches to eval and back on every step): no recomputation
    assert m._eval_stats() is s2
    m.train()
    m.eval()
    assert m._eval_stats() is not s2


def test_deferred_conv_not_for_more_offsets_than_the_tensor_core_wgrad_takes():
    """A 5x5x5 layer (125 offsets) runs on the SIMT kernels, so its eval forward is not deferred to the tensor-core
    inference epilogue either; 3x3x3 and 2x2x2 layers are."""
    from lidog_b200.me import conv
    ok = dict(training=False, grad_enabled=False, has_bias=False, cin=32, cout=64, is_cuda=True, n_out=1000)
    for kv in (1, 8, 27, conv.TC_MAX_KERNEL_VOLUME):
        assert conv.infer_fast_path(**ok, kernel_volume=kv), kv
    assert not conv.infer_fast_path(**ok, kernel_volume=125)
