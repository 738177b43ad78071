"""Per-scan covariance kernels (lg_inst_cov_forward / _backward) against torch formulations of the same op.

    python tools/isw_bench.py [--iters 50] [--warmup 5]

Shapes: the rows of the KITTI-shaped batch of 8 scans (lidog/synth.py, voxel 0.05, the training bench's batch) at
tensor stride 1 with 32 channels and at tensor stride 8 with 128 channels -- the two ends of MinkUNet34's encoder.
Features are seeded normal values; rows keep the batch order of the voxeliser.

Timing: CUDA events around every call, with a 512 MB buffer overwritten before each one, so no input is read from the
126 MB L2; `*_ms` are medians.  The library calls go through the C ABI.  Two torch formulations are timed forward
and forward + backward (autograd, gradient of a sum of the covariances weighted by a random G):
  - `torch_loop`: a Python loop over scans, `x[bidx == b]` then `f^T f / (n_b - 1) + eps I` -- one host
    synchronisation per scan (the boolean index);
  - `torch_padded`: rows scattered into a zero-padded [B, max n_b, C] tensor, one `bmm` -- the counts and the row
    positions are computed on the device, the padded size needs one host read.
Bounds: bytes are the algorithmic ones (forward reads x and the batch index, writes cov; backward reads x and the
batch index, writes dx); FMAs forward n C (C + 1) / 2 (the upper triangle), backward n C^2.  The HBM bound uses the
data-sheet 7.7 TB/s; the FP32 bound is 148 SMs x 128 FMA per clock at the maximum SM clock read in the same run.
`share_*` = bound time / measured time.  Prints one JSON line with the device name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBM_BW = 7.7e12


def _device_facts(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=60).stdout
        name, power, clock = [s.strip() for s in out.strip().split(",")]
        return dict(device=name, power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except Exception as e:
        return dict(device=None, power_limit_w=None, max_sm_clock_mhz=None, device_query_error=str(e))


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
    from lidog_b200.me.isw import COVARIANCE_EPS as EPS

    if not torch.cuda.is_available():
        raise SystemExit("isw_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    L = cabi.lib()
    facts = _device_facts(0)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    fma_rate = sms * 128 * (facts["max_sm_clock_mhz"] or 0) * 1e6  # FP32 FMA per second
    scans = synth.make_batch(8, shape="kitti")
    pts = [torch.from_numpy(p).to(dev) for p, _ in scans]
    cm = ME.CoordinateManager.from_quantized(ME.utils.sparse_quantize_batch(pts, None, 0.05))
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = cabi.stream_of(flush)

    def timed(fn, iters=args.iters):
        for _ in range(args.warmup):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    out = dict(tool="isw_bench", **facts, sm_count=sms, iters=args.iters, levels=[])
    g = torch.Generator(device=dev).manual_seed(0)
    for ts, C in ((1, 32), (8, 128)):
        coords = cm.get_coords(ts).contiguous()
        n = coords.shape[0]
        B = int(coords[:, 0].max()) + 1
        x = torch.randn(n, C, device=dev, generator=g)
        G = torch.randn(B, C, C, device=dev, generator=g)
        cov = torch.empty(B, C, C, device=dev)
        counts = torch.empty(B, dtype=torch.int32, device=dev)
        dx = torch.empty_like(x)

        def fwd():
            cabi.check(L.lg_inst_cov_forward(x.data_ptr(), coords.data_ptr(), n, C, B, EPS, cov.data_ptr(),
                                             counts.data_ptr(), stream))

        def bwd():
            cabi.check(L.lg_inst_cov_backward(x.data_ptr(), coords.data_ptr(), n, C, B, G.data_ptr(),
                                              counts.data_ptr(), dx.data_ptr(), stream))

        bidx = coords[:, 0].long()
        eye = torch.eye(C, device=dev)

        def loop_cov(xx):
            res = []
            for b in range(B):
                f = xx[bidx == b]
                res.append(f.t() @ f / (f.shape[0] - 1) + EPS * eye)
            return torch.stack(res)

        def padded_cov(xx):
            cnt = torch.bincount(bidx, minlength=B)
            start = torch.cumsum(cnt, 0) - cnt
            order = torch.argsort(bidx, stable=True)
            pos = torch.arange(n, device=dev) - start[bidx[order]]
            P = torch.zeros(B, int(cnt.max()), C, device=dev)
            P = P.index_put((bidx[order], pos), xx[order])
            return torch.bmm(P.transpose(1, 2), P) / (cnt - 1).clamp_min(1).view(B, 1, 1) + EPS * eye

        fwd()
        bwd()
        torch.cuda.synchronize()
        xd = x.double()
        ref = loop_cov(xd)
        err = float((cov.double() - ref).norm() / ref.norm())
        xg = xd.clone().requires_grad_(True)
        (loop_cov(xg) * G.double()).sum().backward()
        derr = float((dx.double() - xg.grad).norm() / xg.grad.norm())
        f_ms, b_ms = timed(fwd), timed(bwd)
        level = dict(tensor_stride=ts, rows=n, channels=C, scans=B, fwd_ms=round(f_ms, 4), bwd_ms=round(b_ms, 4))
        f_bytes, b_bytes = 4 * n * C + 4 * n + 4 * B * C * C, 8 * n * C + 4 * n + 4 * B * C * C
        f_fma, b_fma = n * C * (C + 1) // 2, n * C * C
        for name, ms, nbytes, fma in (("fwd", f_ms, f_bytes, f_fma), ("bwd", b_ms, b_bytes, b_fma)):
            hbm_ms, fp32_ms = nbytes / HBM_BW * 1e3, (fma / fma_rate * 1e3 if fma_rate else None)
            level.update({f"{name}_dram_bytes": nbytes, f"{name}_fma": fma,
                          f"{name}_share_hbm": round(hbm_ms / ms, 3),
                          f"{name}_share_fp32": round(fp32_ms / ms, 3) if fp32_ms else None})
        for tname, fn in (("torch_loop", loop_cov), ("torch_padded", padded_cov)):
            def t_fwd(fn=fn):
                with torch.no_grad():
                    fn(x)

            xt = x.clone().requires_grad_(True)

            def t_fwdbwd(fn=fn, xt=xt):
                (fn(xt) * G).sum().backward()

            level[f"{tname}_fwd_ms"] = round(timed(t_fwd, min(args.iters, 20)), 4)
            level[f"{tname}_fwd_bwd_ms"] = round(timed(t_fwdbwd, min(args.iters, 20)), 4)
        level.update(rel_err_cov_vs_fp64=err, rel_err_dx_vs_fp64=derr)
        out["levels"].append(level)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
