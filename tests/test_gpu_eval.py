"""GPU: the evaluation path -- the inference epilogue of the tensor-core convolution (lg_conv_layer_infer), the device
confusion matrix (lg_confusion_matrix), the eval-mode model forward built on them, and LidogEvaluator."""
import numpy as np
import pytest
import torch

from tests.helpers import random_voxels, record

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------- layer: bit-exact
def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _layer_setup(cuda, kind, ts_in, ksize, cin, cout, n_vox, seed):
    import MinkowskiEngine as ME
    rng = np.random.default_rng(seed)
    coords = random_voxels(rng, n_vox, span=30 if n_vox > 500 else 6)
    base = ME.SparseTensor(coordinates=torch.from_numpy(coords).to(cuda), features=torch.ones(len(coords), 1, device=cuda))
    cm = base.coordinate_manager
    for ts in (1, 2, 4, 8):
        cm.get_coords(ts)
    torch.manual_seed(seed)
    cls = ME.MinkowskiConvolutionTranspose if kind == "up" else ME.MinkowskiConvolution
    layer = cls(cin, cout, kernel_size=ksize, stride=2 if kind in ("down", "up") else 1, dimension=3).to(cuda)
    ts_out, plans = layer._plans(cm, ts_in)
    return cm, layer, ts_out, plans[0]


def _without_tiles(plan, every=3):
    """The same plan with the offsets of every `every`-th tile removed: those tiles have no neighbour at all."""
    from lidog_b200.me.coords import GatherPlan
    mask = plan.tile_mask.clone()
    mask[::every] = 0
    return GatherPlan(plan.nbr, plan.k_stride, plan.out_row, mask, plan.K, plan.n_slots, plan.n_out, plan.n_in)


def _bn_stats(C, gen, device):
    mean = torch.randn(C, generator=gen)
    invstd = torch.rand(C, generator=gen) + 0.5
    scale = torch.randn(C, generator=gen) * 0.7 + 0.8  # some negative: the ReLU sees both signs of the shift
    shift = torch.randn(C, generator=gen) * 0.5
    return torch.cat([mean, invstd, scale, shift]).float().to(device)


class _Layer:
    """One layer's operands and the two ways to compute conv -> BN (eval) [-> + res] [-> ReLU]."""

    def __init__(self, plan, cin, cout, kernel, fmt, device, gen):
        from lidog_b200.me import conv as meconv
        self.plan, self.cin, self.cout, self.fmt = plan, cin, cout, fmt
        self.x = torch.randn(plan.n_in, cin, generator=gen).relu_().to(device)
        self.x16 = meconv._cast16(self.x, fmt)
        self.W = kernel.detach().contiguous()
        dt = meconv._dt16(fmt)
        self.w16 = torch.empty((plan.K, cin, cout), dtype=dt, device=device)
        self.w16t = torch.empty((plan.K, cout, cin), dtype=dt, device=device)
        self.st = _bn_stats(cout, gen, device)
        self.dt = dt

    def _out(self):
        n = self.plan.n_out
        y = torch.full((n, self.cout), float("nan"), device=self.x.device)
        return y, torch.full((n, self.cout), -1, dtype=torch.int16, device=self.x.device).view(self.dt)

    def composed(self, res, relu):
        from lidog_b200 import cabi
        L, s = cabi.lib(), cabi.stream_of(self.x)
        y0 = torch.full((self.plan.n_out, self.cout), float("nan"), device=self.x.device)
        cabi.check(L.lg_conv_layer_forward(self.plan.cref, self.x16.data_ptr(), self.cin, self.W.data_ptr(), self.cout,
                                           self.w16.data_ptr(), self.w16t.data_ptr(), 1, self.fmt, None,
                                           y0.data_ptr(), None, s), "lg_conv_layer_forward")
        y, y16 = self._out()
        cabi.check(L.lg_bn_apply(y0.data_ptr(), self.st.data_ptr(), None, None, cabi.ptr(res), relu, self.plan.n_out,
                                 self.cout, y.data_ptr(), y16.data_ptr(), self.fmt, s), "lg_bn_apply")
        return y, y16

    def fused(self, res, relu, prep=0):
        from lidog_b200 import cabi
        y, y16 = self._out()
        cabi.check(cabi.lib().lg_conv_layer_infer(self.plan.cref, self.x16.data_ptr(), self.cin, self.W.data_ptr(),
                                                  self.cout, self.w16.data_ptr(), self.w16t.data_ptr(), prep, self.fmt,
                                                  self.st.data_ptr(), cabi.ptr(res), relu, y.data_ptr(),
                                                  y16.data_ptr(), cabi.stream_of(self.x)), "lg_conv_layer_infer")
        return y, y16


def _check_layer(cuda, kind, ts_in, ksize, cin, cout, n_vox=9000, seed=0, mask_every=0, fmt_name="fp16"):
    from lidog_b200 import cabi
    from lidog_b200.me import conv as meconv
    fmt = cabi.FMT_FP16 if fmt_name == "fp16" else cabi.FMT_BF16
    cm, layer, ts_out, plan = _layer_setup(cuda, kind, ts_in, ksize, cin, cout, n_vox, seed)
    if mask_every:
        plan = _without_tiles(plan, mask_every)
    gen = torch.Generator().manual_seed(seed)
    lay = _Layer(plan, cin, cout, layer.kernel, fmt, cuda, gen)
    # a residual that is itself conv + BN (the block's downsample): a 1x1 layer on the output map
    plan_id = cm.plan("identity", ts_out, ts_out, 1)
    down = _Layer(plan_id, 64, cout, torch.randn(64, cout, generator=gen).to(cuda) * 0.1, fmt, cuda, gen)
    res_bn, _ = down.fused(None, 0, prep=1)
    ref_bn, _ = down.composed(None, 0)
    assert torch.equal(_bits(res_bn), _bits(ref_bn))
    residuals = {"none": None, "plain": torch.randn(plan.n_out, cout, generator=gen).to(cuda), "conv_bn": res_bn}
    n_cases = 0
    for res_name, res in residuals.items():
        for relu in (0, 1):
            y_ref, y16_ref = lay.composed(res, relu)
            y, y16 = lay.fused(res, relu)
            y2, y16_2 = lay.fused(res, relu)
            what = (kind, ts_in, cin, cout, n_vox, mask_every, fmt_name, res_name, relu)
            assert not torch.isnan(y_ref).any(), what
            assert torch.equal(_bits(y), _bits(y_ref)), what
            assert torch.equal(_bits(y16), _bits(y16_ref)), what
            assert torch.equal(_bits(y2), _bits(y)) and torch.equal(_bits(y16_2), _bits(y16)), what  # run to run
            n_cases += 1
    return n_cases


LAYER_CASES = [  # every plan kind of MinkUNet34 and every Cout of its tensor-core layers
    ("same", 1, 3, 32, 32), ("same", 2, 3, 64, 64), ("same", 1, 3, 128, 96), ("same", 2, 3, 96, 128),
    ("same", 4, 3, 256, 256), ("same", 2, 3, 384, 256),
    ("down", 1, 2, 32, 32), ("down", 2, 2, 64, 64), ("down", 4, 2, 128, 128),
    ("up", 2, 2, 256, 128), ("up", 4, 2, 128, 96), ("up", 2, 2, 96, 96), ("up", 8, 2, 256, 256),
    ("identity", 1, 1, 32, 64), ("identity", 2, 1, 384, 256), ("identity", 1, 1, 128, 96),
]


@pytest.mark.parametrize("kind,ts_in,ksize,cin,cout", LAYER_CASES)
def test_conv_layer_infer_bit_identical_to_conv_then_bn_apply(cuda, kind, ts_in, ksize, cin, cout):
    assert _check_layer(cuda, kind, ts_in, ksize, cin, cout) == 6


@pytest.mark.parametrize("n_vox", [1, 100, 200, 300])
@pytest.mark.parametrize("kind,ts_in,ksize,cin,cout", [("same", 1, 3, 64, 64), ("identity", 1, 1, 32, 96),
                                                       ("same", 1, 3, 256, 256)])
def test_conv_layer_infer_small_sets(cuda, n_vox, kind, ts_in, ksize, cin, cout):
    """1-3 tiles: partial tiles, padding rows, super-tiles with fewer tiles than the accumulator set."""
    _check_layer(cuda, kind, ts_in, ksize, cin, cout, n_vox=n_vox, seed=n_vox)


@pytest.mark.parametrize("kind,ts_in,ksize,cin,cout", [("same", 1, 3, 64, 64), ("down", 1, 2, 32, 32),
                                                       ("up", 2, 2, 96, 96), ("identity", 2, 1, 384, 256)])
@pytest.mark.parametrize("every", [1, 3])
def test_conv_layer_infer_tiles_without_neighbours(cuda, kind, ts_in, ksize, cin, cout, every):
    """Tiles with no neighbour at all write act(shift [+ res]), exactly what BN-apply makes of the zeros."""
    _check_layer(cuda, kind, ts_in, ksize, cin, cout, mask_every=every)


@pytest.mark.parametrize("kind,ts_in,ksize,cin,cout", [("same", 1, 3, 96, 96), ("up", 2, 2, 256, 128)])
def test_conv_layer_infer_bf16(cuda, kind, ts_in, ksize, cin, cout):
    _check_layer(cuda, kind, ts_in, ksize, cin, cout, fmt_name="bf16")


# ------------------------------------------------------------------------------------------- confusion matrix
def _np_confusion(logits, target, C):
    pred = np.argmax(logits, 1)  # first maximal index, like torch.argmax
    row = np.where((target >= 0) & (target < C), target, C)
    conf = np.zeros((C + 1, C), dtype=np.int64)
    np.add.at(conf, (row, pred), 1)
    return conf


def _confusion(logits, target, conf):
    from lidog_b200 import cabi
    cabi.check(cabi.lib().lg_confusion_matrix(cabi.ptr(logits), logits.shape[0], conf.shape[1], cabi.ptr(target),
                                              cabi.ptr(conf), cabi.stream_of(conf)), "lg_confusion_matrix")


@pytest.mark.parametrize("C", [7, 19, 32])
def test_confusion_matrix_matches_numpy(cuda, C):
    rng = np.random.default_rng(C)
    conf = torch.zeros((C + 1, C), dtype=torch.int64, device=cuda)
    want = np.zeros((C + 1, C), dtype=np.int64)
    for n in (0, 1, 255, 1025, 300001):  # several calls accumulate; n not a multiple of the block size
        logits = rng.integers(-3, 4, (n, C)).astype(np.float32)  # few values: many ties
        target = rng.integers(-1, C + 2, n).astype(np.int64)    # ignore label and out-of-range targets
        target[rng.random(n) < 0.01] = 255
        _confusion(torch.from_numpy(logits).to(cuda), torch.from_numpy(target).to(cuda), conf)
        want += _np_confusion(logits, target, C)
    assert np.array_equal(conf.cpu().numpy(), want)
    # run to run identical
    logits = torch.randn(200003, C, device=cuda)
    target = torch.randint(-1, C, (200003,), device=cuda)
    a = torch.zeros_like(conf)
    b = torch.zeros_like(conf)
    _confusion(logits, target, a)
    _confusion(logits, target, b)
    assert torch.equal(a, b) and int(a.sum()) == 200003


# ------------------------------------------------------------------------------------------- whole model
def _crop_scan(seed=3):
    from lidog_b200.lidog import synth
    pts, lab = synth.make_scan(seed, "nuscenes")
    keep = (np.abs(pts[:, 0]) < 12) & (np.abs(pts[:, 1]) < 12)
    return pts[keep], lab[keep]


def _rel(a, b):
    return float((a.detach().cpu().double() - b.detach().cpu().double()).norm() / b.detach().cpu().double().norm())


@pytest.fixture(scope="module")
def trained_state(cuda):
    """MinkUNet34BEV with non-trivial running statistics: a few training-mode forwards on the crop (and a second
    crop), then the state dict; plus the crop's voxels."""
    import MinkowskiEngine as ME
    from oracle import voxel as ov
    from lidog_b200.lidog.model import MinkUNet34BEV
    torch.manual_seed(0)
    model = MinkUNet34BEV(1, 7, mapping_bound_2d=12.0).to(cuda)
    model.train()
    with torch.no_grad():
        for seed in (5, 6, 3):
            pts, lab = _crop_scan(seed)
            q, _, _, _, _ = ov.sparse_quantize(pts, np.ones((len(pts), 1), np.float32), lab, -1, True, True, False, 0.05)
            coords = ov.batched_coordinates([q])
            x = ME.SparseTensor(coordinates=torch.from_numpy(coords).to(cuda), features=torch.ones(len(q), 1, device=cuda))
            model(x, is_train=False)
    state = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    assert int(state["bn1.bn.num_batches_tracked"]) == 3
    return dict(state=state, coords=coords, n=len(q), lab=lab)


def _gpu_model(cuda, state):
    from lidog_b200.lidog.model import MinkUNet34BEV
    torch.manual_seed(0)
    m = MinkUNet34BEV(1, 7, mapping_bound_2d=12.0)
    m.load_state_dict(state)
    return m.to(cuda)


def _input(cuda, ts):
    import MinkowskiEngine as ME
    return ME.SparseTensor(coordinates=torch.from_numpy(ts["coords"]).to(cuda),
                           features=torch.ones(ts["n"], 1, device=cuda))


def test_model_eval_forward_matches_oracle(cuda, trained_state):
    from lidog_b200 import cabi
    from lidog_b200.me.conv import DeferredConv
    from oracle import me_cpu
    from oracle.me_cpu.bevfn import sparse2super as o_s2s
    from lidog_b200.lidog.model import MinkUNet34BEV
    ts = trained_state
    torch.manual_seed(0)
    ref = MinkUNet34BEV(1, 7, ME=me_cpu, bev_fn=o_s2s, mapping_bound_2d=12.0)
    ref.load_state_dict(ts["state"])
    ref = ref.double().eval()
    with torch.no_grad():
        xo = me_cpu.SparseTensor(coordinates=torch.from_numpy(ts["coords"]),
                                 features=torch.ones(ts["n"], 1, dtype=torch.float64))
        ref_logits = ref(xo, is_train=False)[0].F
    model = _gpu_model(cuda, ts["state"]).eval()
    # the fast path is really taken: a tensor-core convolution returns a DeferredConv under no_grad in eval mode
    with torch.no_grad():
        probe = model.conv1p1s2(model.relu(model.bn0(model.conv0p1s1(_input(cuda, ts)))))
        assert isinstance(probe, DeferredConv)
        cabi.counting(True)
        try:
            fast = model(_input(cuda, ts), is_train=False)[0].F
            counts = dict(cabi.COUNTS)
            launches = cabi.kernel_launches()
        finally:
            cabi.counting(False)
    assert counts.get("lg_conv_layer_infer", 0) == 61, counts
    # the layer calls of the training path report their launches through count_launches ("#" + name)
    assert "#lg_conv_layer_forward" not in counts and "#lg_bn_layer_forward" not in counts, counts
    assert counts.get("lg_cast_rows", 0) == 1, counts  # only the stem's output is cast; Y16 feeds every other layer
    today = model(_input(cuda, ts), is_train=False)[0].F.detach()  # eval with autograd on: today's path
    err_fast = _rel(fast, ref_logits)
    err_today = _rel(today, ref_logits)
    diff = _rel(fast, today)
    agree = float((fast.argmax(1) == today.argmax(1)).float().mean())
    agree_ref = float((fast.argmax(1).cpu() == ref_logits.argmax(1)).float().mean())
    record("eval_forward", voxels=ts["n"], logits_vs_f64=err_fast, today_vs_f64=err_today, fast_vs_today=diff,
           argmax_agree_today=agree, argmax_agree_f64=agree_ref, library_calls=counts, kernel_launches=launches)
    assert err_fast <= 4e-3, err_fast
    assert err_today <= 4e-3, err_today
    assert agree >= 0.99, agree


def test_eval_pass_has_no_side_effects(cuda, trained_state):
    from lidog_b200.lidog import losses
    ts = trained_state
    sem = torch.from_numpy(np.zeros(ts["n"], np.int64)).to(cuda)
    sem[::3] = 2
    sem[1::3] = 5

    def train_step(model):
        model.train()
        model.zero_grad(set_to_none=True)
        out, bev = model(_input(cuda, ts), is_train=True)
        loss = losses.soft_dice_loss(out.F, sem, -1) + bev["block8"].square().mean()
        loss.backward()
        return loss.detach(), {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}

    old_det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        a = _gpu_model(cuda, ts["state"])
        before = {k: v.detach().clone() for k, v in a.state_dict().items()}
        a.eval()
        with torch.no_grad():
            a(_input(cuda, ts), is_train=False)
        after = a.state_dict()
        for k, v in before.items():
            assert torch.equal(v, after[k]), k  # parameters, running buffers and num_batches_tracked
        loss_a, grads_a = train_step(a)
        b = _gpu_model(cuda, ts["state"])
        loss_b, grads_b = train_step(b)
    finally:
        torch.backends.cudnn.deterministic = old_det
    assert torch.equal(loss_a, loss_b)
    assert grads_a.keys() == grads_b.keys()
    for k in grads_a:
        assert torch.equal(grads_a[k], grads_b[k]), k
    for k, v in a.state_dict().items():  # the training step's buffer updates too
        assert torch.equal(v, b.state_dict()[k]), k


def test_eval_with_grad_still_backpropagates(cuda, trained_state):
    from lidog_b200.me.conv import DeferredConv
    ts = trained_state
    model = _gpu_model(cuda, ts["state"]).eval()
    out, _ = model(_input(cuda, ts), is_train=False)
    assert not isinstance(out, DeferredConv) and out.F.requires_grad
    out.F.square().mean().backward()
    g = model.block1[0].conv1.kernel.grad
    assert g is not None and torch.isfinite(g).all() and float(g.abs().sum()) > 0
    assert model.block1[0].norm1.bn.weight.grad is not None


# ------------------------------------------------------------------------------------------- evaluator
def test_evaluator_matches_sklearn(cuda):
    from sklearn.metrics import jaccard_score
    from lidog_b200.lidog import synth
    from lidog_b200.lidog.evaluate import LidogEvaluator
    from lidog_b200.lidog.model import MinkUNet34BEV
    from tests.refharness import _JaccardIndex
    torch.manual_seed(0)
    model = MinkUNet34BEV(1, 7).to(cuda)
    model.train()
    ev = LidogEvaluator(model, 7, ignore_label=-1)
    all_logits, all_lab = [], []
    for seed in (10, 20):
        scans = synth.make_batch(2, seed, "kitti", 7)
        pts = [torch.from_numpy(p).to(cuda) for p, _ in scans]
        lab = [torch.from_numpy(l).to(cuda) for _, l in scans]
        logits = ev.step(pts, lab)
        _, sem = ev.voxelize(pts, lab)[:2]
        all_logits.append(logits.cpu())
        all_lab.append(sem.cpu())
    assert model.training  # restored
    res = ev.result()
    pred = torch.cat(all_logits).argmax(1).numpy()
    target = torch.cat(all_lab).numpy()
    want = jaccard_score(target, pred, labels=list(range(7)), average=None, zero_division=0)
    assert np.array_equal(res["iou"], want)
    assert res["miou"] == float(want.mean())
    want_ig = _JaccardIndex(7, ignore_index=-1)(torch.from_numpy(pred), torch.from_numpy(target)).numpy()
    assert np.array_equal(res["iou_ignore"].astype(np.float32), want_ig)
    assert int(res["confusion"].sum()) == len(target)
    record("evaluator", voxels=int(len(target)), miou=res["miou"], miou_ignore=res["miou_ignore"])
