"""BEV projection kernels at the training bench's shape: `lg_bev_forward` and `lg_bev_backward`.

    python tools/bev_bench.py [--iters 50] [--warmup 5] [--pool 5,3,1] [--bound 50] [--voxel 0.05] [--dense]
    python tools/bev_bench.py --profile-step FILE     # kernel list of one training step instead

Shape: the KITTI-shaped batch of 8 scans the training bench uses (`synth.make_batch(8, 1234, "kitti", 7)`, voxel 0.05),
at tensor stride 1 with 96 channels -- the width of the trunk output the BEV head projects -- onto the 2000 x 2000
image, pooled 5/3/1 to 666 x 666, policy LAST, channels_last output and gradient (what the bench runs).  Features are
seeded post-ReLU normal values, the output gradient seeded normal values.  `--pool K,S,P`, `--bound` and `--voxel`
change the pooling and the image (e.g. `--pool 5,1,1` is the reference's scaling factor 2 or 3, a 1998 x 1998 output).

Timing: CUDA events around every call, with a 512 MB buffer overwritten before each one, so no input is read from the
126 MB L2; `*_ms` are medians.  Each call is timed as a whole, memsets included.  `grad_feats_bytes` (n x C x 4) is
the write every backward must make; `bwd_frac_copy_bw_grad_write` sets it against the measured copy bandwidth of
6551.7 GB/s (DESIGN.md section 4), a lower bound on the backward's traffic; `fwd_frac_copy_bw_out_write` does the same
for the forward's output write (`out_bytes`).  `--dense` also times the dense torch formulation at the same geometry:
a zero (B, H, W, C) image, `index_put_` of the features, the raw re-view as (B, C, H, W) and `max_pool2d`, and its
autograd backward (`dense_fwd_ms`, `dense_bwd_ms`).  Prints one JSON line with the device name and power limit read
in the same run.

--profile-step runs the training bench's model and trainer on the same batch: 3 warm-up steps, then one step under
torch.profiler; FILE gets the CUDA kernels of that step sorted by device time.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COPY_BW = 6551.7e9


def _device_facts(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=60).stdout
        name, power, clock = [s.strip() for s in out.strip().split(",")]
        return dict(device=name, power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except Exception as e:
        return dict(device=None, power_limit_w=None, device_query_error=str(e))


def profile_step(path: str, dev) -> None:
    import torch
    from torch.profiler import ProfilerActivity, profile
    from lidog_b200.lidog import bev as lbev, model as M, step, synth

    torch.backends.cudnn.benchmark = True
    torch.manual_seed(1234)
    net = M.MinkUNet34BEV(1, 7, mapping_bound_2d=synth.SHAPES["kitti"]["bound"]).to(dev)
    if lbev.CONFIG["channels_last"]:
        net.encoders2d.to(memory_format=torch.channels_last)
    trainer = step.LidogTrainer(net, num_classes=7, shape="kitti")
    scans = synth.make_batch(8, 1234, "kitti", 7)
    pts = [torch.from_numpy(p).to(dev) for p, _ in scans]
    lab = [torch.from_numpy(l).to(dev) for _, l in scans]
    for _ in range(3):
        trainer.training_step(pts, lab)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        trainer.training_step(pts, lab)
        torch.cuda.synchronize()
    facts = _device_facts(0)
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=70)
    with open(path, "w") as f:
        f.write(f"# one training step, KITTI batch 8, under torch.profiler; {json.dumps(facts)}\n{table}\n")
    print(table)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--profile-step", metavar="FILE")
    ap.add_argument("--pool", default="5,3,1", help="MaxPool2d kernel,stride,padding")
    ap.add_argument("--bound", type=float, default=None, help="BEV bound in metres (default: the KITTI shape's)")
    ap.add_argument("--voxel", type=float, default=0.05, help="BEV pixel size in metres")
    ap.add_argument("--dense", action="store_true", help="also time the dense torch formulation")
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    from lidog_b200 import cabi
    from lidog_b200 import me as ME
    from lidog_b200.lidog import synth
    from lidog_b200.lidog.bev import image_size

    if not torch.cuda.is_available():
        raise SystemExit("bev_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    if args.profile_step:
        profile_step(args.profile_step, dev)
        return
    L = cabi.lib()
    scans = synth.make_batch(8, 1234, "kitti", 7)
    res = ME.utils.sparse_quantize_batch([torch.from_numpy(p).to(dev) for p, _ in scans], None, 0.05)
    coords = ME.CoordinateManager.from_quantized(res).get_coords(1).contiguous()
    n, C, B = coords.shape[0], 96, 8
    bound = synth.SHAPES["kitti"]["bound"] if args.bound is None else args.bound
    vs = args.voxel
    H = W = image_size(bound, vs)
    pk, ps, pp = (int(v) for v in args.pool.split(","))
    h, w = (H + 2 * pp - pk) // ps + 1, (W + 2 * pp - pk) // ps + 1
    g = torch.Generator(device=dev).manual_seed(0)
    feats = torch.randn(n, C, device=dev, generator=g).clamp_min_(0)
    grad_out = torch.randn(B, C, h, w, device=dev, generator=g).contiguous(memory_format=torch.channels_last)
    out = torch.empty((B, C, h, w), device=dev).contiguous(memory_format=torch.channels_last)
    grad_feats = torch.empty(n, C, device=dev)
    ws_bytes = L.lg_bev_workspace(n, C, B, H, W, pk, ps, pp)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = cabi.stream_of(flush)

    def fwd():
        cabi.check(L.lg_bev_forward(coords.data_ptr(), feats.data_ptr(), n, C, B, float(bound), vs, H, W, pk, ps, pp,
                                    cabi.BEV_LAST, 1, out.data_ptr(), ws.data_ptr(), ws_bytes, stream))

    def bwd():
        cabi.check(L.lg_bev_backward(coords.data_ptr(), feats.data_ptr(), n, C, B, H, W, pk, ps, pp, cabi.BEV_LAST, 1,
                                     grad_out.data_ptr(), grad_feats.data_ptr(), ws.data_ptr(), ws_bytes, stream))

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        ts = []
        for _ in range(args.iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts), min(ts), max(ts)

    f_ms, f_min, f_max = timed(fwd)
    b_ms, b_min, b_max = timed(bwd)  # the workspace holds what the last forward recorded
    gbytes, obytes = n * C * 4, B * C * h * w * 4
    extra = {}
    if args.dense:
        del out, ws
        torch.cuda.empty_cache()
        extra = _time_dense(timed, coords, feats, B, bound, vs, H, (pk, ps, pp), grad_out)
    print(json.dumps(dict(
        tool="bev_bench", **_device_facts(0), iters=args.iters, rows=n, channels=C, batch=B, image=H, pooled=h,
        pool=[pk, ps, pp], bound=bound, voxel=vs, workspace_bytes=ws_bytes, fwd_ms=round(f_ms, 4),
        fwd_ms_min=round(f_min, 4), fwd_ms_max=round(f_max, 4), bwd_ms=round(b_ms, 4), bwd_ms_min=round(b_min, 4),
        bwd_ms_max=round(b_max, 4), grad_feats_bytes=gbytes,
        bwd_frac_copy_bw_grad_write=round(gbytes / (b_ms * 1e-3) / COPY_BW, 3),
        out_bytes=obytes, fwd_frac_copy_bw_out_write=round(obytes / (f_ms * 1e-3) / COPY_BW, 3), **extra)))


def _time_dense(timed, coords, feats, B, bound, vs, H, pool, grad_out) -> dict:
    """The dense torch formulation of the same projection, batched (no per-sample loop or host copy): pixel maths in
    float32 as the reference does it, a zero image, index_put_, the raw re-view, max_pool2d; autograd backward."""
    import torch
    import torch.nn.functional as F
    C = feats.shape[1]
    xyz = coords[:, 1:3].float() * vs
    inb = (-bound < xyz[:, 0]) & (xyz[:, 0] < bound) & (-bound < xyz[:, 1]) & (xyz[:, 1] < bound)
    px = torch.floor((xyz[:, 0] - (-bound)) / vs).long()
    py = torch.floor(H - (xyz[:, 1] - (-bound)) / vs).long() - 1
    py = torch.where(py < 0, py + H, py)
    pix = (coords[:, 0].long() * H + py) * H + px
    pix, rows = pix[inb], torch.nonzero(inb)[:, 0]
    f = feats.detach().requires_grad_(True)
    state = {}

    def fwd():
        img = torch.zeros(B * H * H, C, device=feats.device).index_put((pix,), f[rows])
        state["out"] = F.max_pool2d(img.view(B, C, H, H), *pool)

    def bwd():
        torch.autograd.grad(state["out"], f, grad_out, retain_graph=True)

    fm, _, _ = timed(fwd)
    bm, _, _ = timed(bwd)
    return dict(dense_fwd_ms=round(fm, 4), dense_bwd_ms=round(bm, 4))


if __name__ == "__main__":
    main()
