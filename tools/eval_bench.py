"""Eval throughput of MinkUNet34BEV: scans/s of the `model.eval()` forward under `torch.no_grad()`, on the synthetic
KITTI-shaped batch of 8 and nuScenes-shaped batch of 16 scans (lidog/synth.py).  Voxelisation and the confusion-matrix
update (lg_confusion_matrix, where the library has it) are timed separately.

    python tools/eval_bench.py [--tree DIR] [--steps 20] [--warmup 5] [--label NAME] [--dump DIR] [--profile DIR]

The forward uses only the public model / MinkowskiEngine API, so `--tree` can point at another checkout of this
repository (built) and the two are compared with the same file.  Before timing, a few training-mode forwards (no
gradients) give the batch norms non-trivial running statistics; the model and the data are seeded.

Timing: CUDA events around the three phases of every batch (voxelise; forward; metric), after `--warmup` untimed
batches.  The same batch is reused, but it is voxelised again every time, so the forward builds its kernel maps as for
a new scan; `scans_per_s` is the forward alone, `e2e_scans_per_s` voxelisation + forward.  Prints one JSON line with
the device name and power limit read in the same run.  `--dump DIR` writes the logits of the first batch of each shape
(`eval_logits_<shape>.npy`); `--profile DIR` runs one eval forward per shape under torch.profiler and writes the
kernel list (`eval_kernels_<label>_<shape>.txt`), with the launch count in the JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _device_facts(index: int) -> dict:
    """Name, power limit and max SM clock of the card, from nvidia-smi (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=60).stdout
        name, power, clock = [s.strip() for s in out.strip().split(",")]
        return dict(device=name, power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except Exception as e:  # the numbers are reported without them rather than not at all
        return dict(device=None, power_limit_w=None, device_query_error=str(e))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT, help="repository checkout whose lidog_b200 is measured")
    ap.add_argument("--label", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--classes", type=int, default=7)
    ap.add_argument("--shapes", default="kitti:8,nuscenes:16")
    ap.add_argument("--dump", default=None)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if args.steps < 20:
        raise SystemExit("--steps must be >= 20")
    tree = os.path.abspath(args.tree)
    sys.path.insert(0, tree)
    import numpy as np
    import torch
    from lidog_b200 import cabi
    from lidog_b200 import me as ME
    from lidog_b200.lidog import model as M
    from lidog_b200.lidog import synth

    if not torch.cuda.is_available():
        raise SystemExit("eval_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    L = cabi.lib()
    has_metric = hasattr(L, "lg_confusion_matrix")
    result = dict(bench="eval_forward", tree=args.label or tree, **_device_facts(0), torch=torch.__version__,
                  steps=args.steps, warmup=args.warmup, classes=args.classes, shapes={})

    for spec in args.shapes.split(","):
        shape, batch = spec.split(":")
        batch = int(batch)
        cfg = synth.SHAPES[shape]
        torch.manual_seed(1234)
        net = M.MinkUNet34BEV(1, args.classes, mapping_bound_2d=cfg["bound"]).to(dev)
        scans = synth.make_batch(batch, 1234, shape, args.classes)
        pts = [torch.from_numpy(p).to(dev) for p, _ in scans]
        lab = [torch.from_numpy(l).to(dev) for _, l in scans]

        def voxelize():
            q = ME.utils.sparse_quantize_batch(pts, lab, 0.05, -1)
            sem = torch.cat(lab, 0)[q["unique_map"]].long()
            cm = ME.CoordinateManager.from_quantized(q)
            cm.batch_size = batch
            x = ME.SparseTensor(features=torch.ones((q["coords"].shape[0], 1), device=dev), coordinate_manager=cm)
            return x, sem

        def run(x):
            return net(x, is_train=False)[0].F

        def forward():
            x, sem = voxelize()
            return run(x), sem

        with torch.no_grad():
            net.train()
            for _ in range(3):  # non-trivial running statistics
                forward()
            net.eval()
            conf = torch.zeros((args.classes + 1, args.classes), dtype=torch.int64, device=dev)

            def metric(logits, sem):
                if has_metric:
                    cabi.check(L.lg_confusion_matrix(logits.data_ptr(), logits.shape[0], args.classes, sem.data_ptr(),
                                                     conf.data_ptr(), cabi.stream_of(logits)), "lg_confusion_matrix")

            logits, sem = forward()
            if args.dump:
                os.makedirs(args.dump, exist_ok=True)
                np.save(os.path.join(args.dump, f"eval_logits_{shape}.npy"), logits.float().cpu().numpy())
            for _ in range(args.warmup):
                metric(*forward())
            torch.cuda.synchronize()
            ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
            for e in ev:
                e[0].record()
                x, sem = voxelize()
                e[1].record()
                logits = run(x)
                e[2].record()
                metric(logits, sem)
                e[3].record()
            torch.cuda.synchronize()
            vox_ms = [e[0].elapsed_time(e[1]) for e in ev]
            fwd_ms = [e[1].elapsed_time(e[2]) for e in ev]
            met_ms = [e[2].elapsed_time(e[3]) for e in ev]
            entry = dict(batch=batch, voxels=int(logits.shape[0]), scans_per_s=batch * args.steps / (sum(fwd_ms) / 1e3),
                         forward_ms_mean=float(np.mean(fwd_ms)), forward_ms_min=float(np.min(fwd_ms)),
                         forward_ms_max=float(np.max(fwd_ms)), voxelize_ms_mean=float(np.mean(vox_ms)),
                         e2e_scans_per_s=batch * args.steps / ((sum(fwd_ms) + sum(vox_ms)) / 1e3),
                         metric_ms_mean=float(np.mean(met_ms)) if has_metric else None)
            if args.profile:
                from torch.profiler import ProfilerActivity, profile
                os.makedirs(args.profile, exist_ok=True)
                x, _ = voxelize()
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:  # the model forward alone
                    run(x)
                    torch.cuda.synchronize()
                kern = {}
                for e in prof.events():
                    if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy") \
                            and not e.name.startswith("Memset"):
                        k = kern.setdefault(e.name, [0, 0.0])
                        k[0] += 1
                        k[1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                rows = sorted(kern.items(), key=lambda kv: -kv[1][1])
                entry["profile_kernel_launches"] = sum(v[0] for v in kern.values())
                entry["profile_kernels_distinct"] = len(kern)
                label = args.label or os.path.basename(tree)
                with open(os.path.join(args.profile, f"eval_kernels_{label}_{shape}.txt"), "w") as f:
                    f.write(f"# one eval forward (model only, no_grad; kernel maps built inside), {shape} batch {batch}, tree {label}\n")
                    f.write(f"# {result['device']}, power limit {result['power_limit_w']} W; "
                            f"{entry['profile_kernel_launches']} kernel launches\n")
                    f.write(f"{'launches':>8}  {'total_us':>10}  kernel\n")
                    for name, (n, t) in rows:
                        f.write(f"{n:>8}  {t:>10.1f}  {name[:160]}\n")
            result["shapes"][shape] = entry
        del net
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
