"""MinkowskiInstanceNorm (+ ReLU) kernels, forward and backward, against a torch `index_add` formulation.

    python tools/instnorm_bench.py [--iters 50] [--warmup 5]

Shapes: the rows of the KITTI-shaped batch of 8 scans (lidog/synth.py, voxel 0.05, the training bench's batch) at
tensor stride 1 with 32 channels and at tensor stride 8 with 128 channels -- the two ends of MinkUNet34's encoder.
Features are seeded normal values; rows keep the batch order of the voxeliser.

Timing: CUDA events around every call, with a 512 MB buffer overwritten before each one, so neither input is read from
the 126 MB L2; `*_ms` are medians.  `lg_instnorm_forward` / `lg_instnorm_backward` are called through the C ABI; the
torch formulation (per-instance sums by `index_add_`, gathers by index; float atomics, so not deterministic) is timed
forward under `no_grad` and forward + backward under autograd.  DRAM bytes are the algorithmic ones (module docstring
of csrc/instnorm.cu): forward 14 B per element + 8 B per row, backward 28 B per element + 8 B per row; `frac_copy_bw`
is bytes / time over the measured copy bandwidth of 6551.7 GB/s (DESIGN.md section 4).  Prints one JSON line with the
device name and power limit read in the same run.
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


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    from lidog_b200 import cabi
    from lidog_b200 import me as ME
    from lidog_b200.lidog import synth
    from lidog_b200.me.norm import INSTANCE_NORM_EPS as EPS

    if not torch.cuda.is_available():
        raise SystemExit("instnorm_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    L = cabi.lib()
    scans = synth.make_batch(8, shape="kitti")
    pts = [torch.from_numpy(p).to(dev) for p, _ in scans]
    res = ME.utils.sparse_quantize_batch(pts, None, 0.05)
    cm = ME.CoordinateManager.from_quantized(res)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = cabi.stream_of(flush)

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
        return statistics.median(ts)

    out = dict(tool="instnorm_bench", **_device_facts(0), iters=args.iters, levels=[])
    g = torch.Generator(device=dev).manual_seed(0)
    for ts, C in ((1, 32), (8, 128)):
        coords = cm.get_coords(ts).contiguous()
        n = coords.shape[0]
        B = int(coords[:, 0].max()) + 1
        x = torch.randn(n, C, device=dev, generator=g)
        dy = torch.randn(n, C, device=dev, generator=g)
        w = torch.rand(C, device=dev, generator=g) + 0.5
        b = torch.randn(C, device=dev, generator=g)
        y, dx = torch.empty_like(x), torch.empty_like(x)
        y16 = torch.empty((n, C), dtype=torch.float16, device=dev)
        st = torch.empty((2, B, C), dtype=torch.float64, device=dev)
        dwb = torch.empty((2, C), device=dev)

        def fwd():
            cabi.check(L.lg_instnorm_forward(x.data_ptr(), coords.data_ptr(), n, C, B, w.data_ptr(), b.data_ptr(), EPS,
                                             1, y.data_ptr(), y16.data_ptr(), cabi.FMT_FP16, st.data_ptr(), stream))

        def bwd():
            cabi.check(L.lg_instnorm_backward(dy.data_ptr(), x.data_ptr(), y.data_ptr(), coords.data_ptr(), n, C, B,
                                              w.data_ptr(), 1, st.data_ptr(), dx.data_ptr(), dwb[0].data_ptr(),
                                              dwb[1].data_ptr(), stream))

        bidx = coords[:, 0].long()

        def torch_in(xx):
            cnt = torch.zeros(B, device=dev).index_add_(0, bidx, torch.ones(n, device=dev)).clamp_min(1)[:, None]
            mean = torch.zeros(B, C, device=dev).index_add_(0, bidx, xx) / cnt
            xc = xx - mean[bidx]
            var = torch.zeros(B, C, device=dev).index_add_(0, bidx, xc * xc) / cnt
            return torch.relu(xc * torch.rsqrt(var + EPS)[bidx] * w + b)

        def torch_fwd():
            with torch.no_grad():
                torch_in(x)

        xg = x.clone().requires_grad_(True)

        def torch_fwdbwd():
            torch_in(xg).backward(dy)

        fwd()
        torch.cuda.synchronize()
        err = float((y - torch_in(x)).norm() / torch_in(x).norm())
        f_ms, b_ms = timed(fwd), timed(bwd)
        tf_ms, tfb_ms = timed(torch_fwd), timed(torch_fwdbwd)
        f_bytes, b_bytes = 14 * n * C + 8 * n, 28 * n * C + 8 * n
        out["levels"].append(dict(
            tensor_stride=ts, rows=n, channels=C, instances=B, fwd_ms=round(f_ms, 4), bwd_ms=round(b_ms, 4),
            fwd_dram_bytes=f_bytes, bwd_dram_bytes=b_bytes,
            fwd_frac_copy_bw=round(f_bytes / (f_ms * 1e-3) / COPY_BW, 3),
            bwd_frac_copy_bw=round(b_bytes / (b_ms * 1e-3) / COPY_BW, 3),
            torch_index_add_fwd_ms=round(tf_ms, 4), torch_index_add_fwd_bwd_ms=round(tfb_ms, 4),
            speedup_fwd=round(tf_ms / f_ms, 2), speedup_fwd_bwd=round(tfb_ms / (f_ms + b_ms), 2),
            rel_err_vs_torch=err))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
