"""Micro-benchmark of the sparse-convolution kernels on a real batch of synthetic scans.

    python tools/conv_bench.py [--batch 8] [--shape kitti] [--fmt fp16] [--reps 5] [--cases all|top]

For each (tensor stride, kernel, Cin, Cout) case it times forward (k_gemm_tc), dgrad and wgrad through the
C ABI with CUDA events and prints: pairs, (tile,k) units, algorithmic TFLOP/s (2*pairs*Cin*Cout), the
dense-equivalent TFLOP/s (2*units*128*Cin*Cout) and SM cycles per (tile,k) unit.  BASELINE configs[3]
(micro-bench sweep) uses the same entry points.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


CASES_ALL = [
    # kind, ts, ksize, cin, cout
    ("same", 1, 3, 32, 32), ("same", 1, 3, 96, 96), ("same", 1, 3, 128, 96), ("same", 2, 3, 64, 64),
    ("same", 2, 3, 96, 96), ("same", 4, 3, 128, 128), ("same", 8, 3, 256, 256), ("same", 8, 3, 384, 256),
    ("same", 16, 3, 256, 256), ("down", 1, 2, 32, 32), ("up", 2, 2, 96, 96), ("identity", 1, 1, 128, 96),
]
CASES_TOP = [("same", 1, 3, 96, 96), ("same", 2, 3, 64, 64), ("same", 8, 3, 256, 256)]
# the 3x3x3 layer shapes MinkUNet34 actually runs (Appendix A of SURVEY.md), one per (stride, width)
CASES_NET = [("same", 16, 3, 256, 256), ("same", 8, 3, 256, 256), ("same", 8, 3, 128, 128), ("same", 4, 3, 128, 128),
             ("same", 4, 3, 64, 64), ("same", 2, 3, 96, 96), ("same", 2, 3, 32, 32), ("same", 1, 3, 96, 96)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--shape", default="kitti")
    ap.add_argument("--fmt", default="fp16")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="all")
    ap.add_argument("--only", default="fwd,dgrad,wgrad")
    ap.add_argument("--sorted", default="0,1", help="gather-plan row order: 0 natural, 1 mask-sorted")
    ap.add_argument("--points", type=int, default=0,
                    help="micro-bench sweep (BASELINE configs[3]): use ONE random-plane cloud of this many points "
                         "(10k .. 2M) instead of the batch of synthetic scans")
    args = ap.parse_args()

    from lidog_b200 import cabi
    from lidog_b200 import me as ME
    from lidog_b200.me import conv as meconv
    from lidog_b200.lidog import synth

    dev = torch.device("cuda", 0)
    scans = [synth.make_plane_cloud(args.points, 1234)] if args.points else synth.make_batch(args.batch, 1234, args.shape, 7)
    pts = [torch.from_numpy(p).to(dev) for p, _ in scans]
    lab = [torch.from_numpy(l).to(dev) for _, l in scans]
    q = ME.utils.sparse_quantize_batch(pts, lab, 0.05, -1)
    cm = ME.CoordinateManager.from_quantized(q)
    sm_count, _, _ = cabi.device_info()
    clock_mhz = 1965.0
    fmt = {"fp16": cabi.FMT_FP16, "bf16": cabi.FMT_BF16}[args.fmt]
    dt16 = torch.float16 if args.fmt == "fp16" else torch.bfloat16
    L = cabi.lib()
    only = args.only.split(",")
    for srt in [int(v) for v in args.sorted.split(",")]:
      meconv.CONFIG["sorted"] = srt
      for kind, ts, ks, cin, cout in {"all": CASES_ALL, "top": CASES_TOP, "net": CASES_NET}[args.cases]:
          if srt == 1 and kind in ("up", "identity") and "0" in args.sorted.split(","):
              continue  # these plans have no sorted variant
          cls = ME.MinkowskiConvolutionTranspose if kind == "up" else ME.MinkowskiConvolution
          layer = cls(cin, cout, kernel_size=ks, stride=2 if kind in ("down", "up") else 1, dimension=3)
          ts_out, (p_fwd, p_dgrad, p_wgrad, flip) = layer._plans(cm, ts)
          K = ks ** 3
          pairs = p_fwd.count_pairs()
          mask = p_fwd.tile_mask.view(torch.int32)
          units = int(sum(bin(int(v) & 0xFFFFFFFF).count("1") for v in mask.flatten().tolist()))
          units_d = int(sum(bin(int(v) & 0xFFFFFFFF).count("1") for v in p_dgrad.tile_mask.view(torch.int32).flatten().tolist()))
          x16 = torch.randn(p_fwd.n_in, cin, device=dev).relu_().to(dt16)
          dy16 = (torch.randn(p_fwd.n_out, cout, device=dev)).to(dt16)
          w16 = torch.randn(K, cin, cout, device=dev).to(dt16)
          w16t = w16.transpose(1, 2).contiguous()
          y = torch.empty(p_fwd.n_out, cout, device=dev)
          dx = torch.empty(p_fwd.n_in, cin, device=dev)
          dw = torch.empty(K, cin, cout, device=dev)
          ws_bytes = L.lg_conv_wgrad_tc_workspace(p_wgrad.c, cin, cout)
          ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
          res = {}
          if "fwd" in only:
              res["fwd"] = (timed(lambda: cabi.check(L.lg_conv_gemm_tc(
                  p_fwd.c, cabi.ptr(x16), cin, cabi.ptr(w16t), cout, 0, fmt, None, None, cabi.ptr(y),
                  cabi.stream())), args.reps), units, cin, cout)
          if "dgrad" in only:
              res["dgrad"] = (timed(lambda: cabi.check(L.lg_conv_gemm_tc(
                  p_dgrad.c, cabi.ptr(dy16), cout, cabi.ptr(w16), cin, flip, fmt, None, None, cabi.ptr(dx),
                  cabi.stream())), args.reps), units_d, cout, cin)
          if "wgrad" in only:
              res["wgrad"] = (timed(lambda: cabi.check(L.lg_conv_wgrad_tc(
                  p_wgrad.c, cabi.ptr(x16), cin, cabi.ptr(dy16), cout, fmt, None, cabi.ptr(dw), cabi.ptr(ws),
                  ws_bytes, cabi.stream())), args.reps), units, cin, cout)
          for name, (ms, u, a, b) in res.items():
              alg = 2.0 * pairs * cin * cout / (ms * 1e-3) / 1e12
              dense = 2.0 * u * 128 * cin * cout / (ms * 1e-3) / 1e12
              cyc = ms * 1e-3 * clock_mhz * 1e6 * sm_count / max(u, 1)
              print(json.dumps(dict(case=f"{kind} ts{ts} k{ks} {cin}->{cout}", op=name, sorted=srt, ms=round(ms, 4),
                                    n_out=p_fwd.n_out, pairs=pairs, units=u, density=round(pairs / max(u * 128, 1), 3),
                                    alg_tflops=round(alg, 1), dense_tflops=round(dense, 1),
                                    sm_cycles_per_unit=round(cyc))), flush=True)


if __name__ == "__main__":
    main()
