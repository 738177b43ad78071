#!/usr/bin/env python
"""LiDOG training-step benchmark (BASELINE.json metric: LiDOG train scans/s on B200).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the CPU oracle (MinkowskiEngine-CPU-style restatement)

A step = one pass of the hot path over one batch of synthetic SemanticKITTI-shaped scans:
voxelise (GPU hash) -> coordinate / kernel maps -> MinkUNet34 sparse conv fwd -> BEV projection ->
cuDNN 2D head -> losses -> backward (dgrad / wgrad / BEV bwd) -> Adam.  Workload = BASELINE.json
configs[1] (batch 8 scans per GPU, 7 classes, DDP + SyncBN when N > 1).  One JSON line on stdout.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "lidog_train_scans_per_s"
UNIT = "scans/s"


CONFIG_OF_SHAPE = {"kitti": "configs[1]", "nuscenes": "configs[2]", "mix3d": "configs[4]"}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=8)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--batch", type=int, default=8, help="scans per GPU (BASELINE configs[1]: 8)")
    p.add_argument("--shape", default="kitti", choices=["kitti", "nuscenes", "mix3d"],
                   help="kitti = BASELINE configs[1] (the headline); nuscenes = configs[2] (use --batch 16); "
                        "mix3d = configs[4] (two merged scans per sample)")
    p.add_argument("--classes", type=int, default=7)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-baseline-seconds", type=float, default=30.0)
    p.add_argument("--empty-cache", action="store_true",
                   help="call torch.cuda.empty_cache() before every step, as the reference loop does "
                        "(trainer_lighting_2d.py:147-148, clear_cache_int: 1)")
    p.add_argument("--nccl-ctas", type=int, default=int(os.environ.get("LIDOG_NCCL_CTAS", "0")),
                   help="upper bound on the CTAs of NCCL's all-reduce kernels (0 = NCCL's default, the measured best: "
                        "bounding them to 2-4 cost 7 %% at 2 GPUs, profiles/r02_c_ddp_ab_2gpu.txt)")
    p.add_argument("--no-syncbn", action="store_true",
                   help="diagnostic: DDP without the SyncBN conversion (NOT the reference configuration, train_lidog.py:228)")
    p.add_argument("--same-data", action="store_true",
                   help="diagnostic: every rank trains on rank 0's scans (no load skew between ranks at the SyncBN exchanges)")
    p.add_argument("--ddp-bucket-mb", type=int, default=int(os.environ.get("LIDOG_DDP_BUCKET_MB", "25")),
                   help="DistributedDataParallel bucket_cap_mb (25 = torch default)")
    p.add_argument("--ddp-buffers", choices=["flat", "ddp", "off"], default="flat",
                   help="how rank 0's module buffers (BN running statistics) reach the other ranks before every "
                        "forward: 'ddp' = DistributedDataParallel(broadcast_buffers=True), ~190 tensors one by one; "
                        "'flat' = same semantics, buffers are views of one flat tensor per dtype (2 broadcasts); "
                        "'off' = no broadcast")
    p.add_argument("--ddp-static-graph", type=int, default=0, help="DDP static_graph")
    p.add_argument("--ncu", action="store_true",
                   help="profiling run: 1 warm-up + 1 step between cudaProfilerStart/Stop, no e2e / CPU legs "
                        "(use with ncu --profile-from-start off; numbers printed under ncu are not bench values)")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last of them computed as DIR/<name>.npy: its loss, "
                        "a fixed seeded sample of the updated parameters and of their gradients, and the BN "
                        "buffers (~34 MB); the inputs depend only on the arguments, so two builds can be compared")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.ncu):
        p.error("--dump-outputs needs the timed CUDA path (--impl ours, without --ncu)")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], tf_sustained=d["bf16_tflops_sustained"], tf_burst=d["bf16_tflops"],
                    source="measured")
    # MEASURED_PEAKS.json is driver-written and git-ignored; when this checkout lost it, use the values the
    # driver measured on this pool at the start of round 1 (recorded in SURVEY.md section 0).
    return dict(hbm_gbs=6441.9, tf_sustained=1407.8, tf_burst=1669.9, source="measured (round-1 driver values recorded in SURVEY.md)")


def ncu_traffic():
    """DRAM bytes of one k_gemm2 launch from the committed `ncu --set full` capture (profiles/): read + write.
    The capture is the block8 layer shape (tensor stride 1, 96 -> 96, batch 8 kitti-shaped scans)."""
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_gemm2.txt")))
    if not files:
        return None, None
    txt = open(files[-1]).read()
    tot = 0.0
    for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
        m = re.search(re.escape(key) + r" = ([0-9.]+) (\w+)", txt)
        if not m:
            return None, None
        tot += float(m.group(1)) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[m.group(2)]
    return tot, os.path.basename(files[-1])


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU oracle arm
def oracle_step_fn(shape, classes, crop=None):
    """Builds the CPU-oracle trainer (MinkowskiEngine-CPU-style restatement) and one scan."""
    from lidog_b200.lidog import synth, model as M, step
    from oracle import me_cpu
    from oracle.me_cpu.bevfn import sparse2super as o_s2s
    torch.manual_seed(0)
    cfg = synth.SHAPES[shape]
    net = M.MinkUNet34BEV(1, classes, ME=me_cpu, bev_fn=o_s2s, mapping_bound_2d=cfg["bound"])
    tr = step.LidogTrainer(net, num_classes=classes, shape=shape, ME=me_cpu)
    pts, lab = synth.make_scan(1234, shape, classes)
    full_points = len(pts)
    if crop is not None:
        keep = (np.abs(pts[:, 0]) < crop) & (np.abs(pts[:, 1]) < crop)
        pts, lab = pts[keep], lab[keep]
    P, Lb = [torch.from_numpy(pts)], [torch.from_numpy(lab)]

    def run():
        return float(tr.training_step(P, Lb))
    return run, len(pts), full_points


def run_reference(args):
    """`--impl reference`: the reference's CPU path = the oracle, timed on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    budget = 240.0  # seconds for the whole run
    crop, run, n_pts, full = None, None, 0, 1
    for crop in (None, 25.0, 12.0, 6.0):
        run, n_pts, full = oracle_step_fn(args.shape, args.classes, crop)
        t0 = time.perf_counter(); run(); t1 = time.perf_counter() - t0
        if t1 * (args.steps + max(args.warmup - 1, 0)) <= budget or crop == 6.0:
            break
    for _ in range(max(args.warmup - 1, 0)):
        run()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter(); run(); times.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(times))
    frac = n_pts / full
    value = frac / (ms / 1e3)
    sample = (f"1 {args.shape}-shaped scan per step" + ("" if crop is None else f", cropped to |x|,|y|<{crop} m") +
              f" ({n_pts} of {full} points; value = point fraction / step time)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 0, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"LiDOG MinkUNet34BEV training step, synthetic {args.shape}-shaped scans, "
                                   f"{args.classes} classes (BASELINE {CONFIG_OF_SHAPE[args.shape]})", "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline(args):
    """The oracle port timed on this box's host cores, on a bounded sample of the same workload: the UNCROPPED scan when
    one training step of it fits the budget (it does on the 16-core GPU hosts: ~4 s), else a 25 m crop."""
    cores = os.cpu_count() or 1
    old = torch.get_num_threads()
    torch.set_num_threads(cores)
    try:
        for crop in (None, 25.0):
            run, n_pts, full = oracle_step_fn(args.shape, args.classes, crop)
            t0 = time.perf_counter(); run(); first = time.perf_counter() - t0
            if first <= args.cpu_baseline_seconds / 3 or crop is not None:
                break
        times = [first]
        while sum(times) < args.cpu_baseline_seconds and len(times) < 4:
            t0 = time.perf_counter(); run(); times.append(time.perf_counter() - t0)
        t = float(np.median(times[1:] if len(times) > 1 else times))
        frac = n_pts / full
        return {"value": frac / t, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"CPU oracle (ME-CPU-style per-offset index_select/mm/index_add), {len(times)} training "
                          f"step(s) on 1 {args.shape}-shaped scan, {args.classes} classes" +
                          ("" if crop is None else f", cropped to |x|,|y|<{crop} m") +
                          f" ({n_pts} of {full} points, value = point fraction / median step time {t:.2f} s)"}
    finally:
        torch.set_num_threads(old)


# ------------------------------------------------------------------------------------------ CUDA arm
DUMP_SAMPLE = 1 << 22  # elements kept of the parameter and gradient vectors: 2 x 16 MB of float32


def dump_outputs(path, model, loss):
    """What one training step hands its caller, as float32 / float64 .npy files under `path`:
    loss.npy        the total loss the step returned
    parameters.npy  the parameters after the Adam step  } all parameters flattened in named_parameters() order,
    gradients.npy   the gradients that step applied     } then the same fixed seeded sample of DUMP_SAMPLE elements
                    (zero for a parameter the step gave no gradient)
    buffers.npy     every buffer (BN running statistics, batch counters) flattened in named_buffers() order, float64"""
    os.makedirs(path, exist_ok=True)
    params = [p for _, p in model.named_parameters()]
    n = sum(p.numel() for p in params)
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(DUMP_SAMPLE, n), replace=False))
    idx = torch.from_numpy(idx).to(params[0].device)
    out = {"loss": loss.detach().float().cpu().numpy(),
           "parameters": torch.cat([p.detach().reshape(-1) for p in params])[idx].float().cpu().numpy(),
           "gradients": torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1)
                                   for p in params])[idx].float().cpu().numpy(),
           "buffers": torch.cat([b.detach().reshape(-1).double() for _, b in model.named_buffers()]).cpu().numpy()}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    import torch.distributed as dist
    from lidog_b200 import cabi
    from lidog_b200.lidog import synth, model as M, step
    from lidog_b200 import me as ME
    from lidog_b200.me import conv as meconv
    from lidog_b200.me import norm as menorm
    from lidog_b200.me import peer as mepeer
    from lidog_b200.me import coords as mecoords

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the oracle")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        opts = None
        if args.nccl_ctas > 0:
            try:
                opts = dist.ProcessGroupNCCL.Options()
                opts.config.max_ctas = args.nccl_ctas
                opts.config.min_ctas = 1
            except Exception:
                opts = None
                os.environ.setdefault("NCCL_MAX_CTAS", str(args.nccl_ctas))
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    cabi.lib()
    torch.backends.cudnn.benchmark = True  # train_lidog.py:312

    cfg = synth.SHAPES[args.shape]
    torch.manual_seed(1234)
    net = M.MinkUNet34BEV(1, args.classes, mapping_bound_2d=cfg["bound"]).to(dev)
    from lidog_b200.lidog import bev as lbev
    if lbev.CONFIG["channels_last"]:  # 4-D (2D-head) parameters only; the logical shapes do not change
        net.encoders2d.to(memory_format=torch.channels_last)
    if world > 1:  # train_lidog.py:227-231
        if not args.no_syncbn:
            net = ME.MinkowskiSyncBatchNorm.convert_sync_batchnorm(net)
        # gradient_as_bucket_view: the all-reduce works on the gradient storage itself (no bucket copies); same result
        from lidog_b200.lidog import ddp as lddp
        ddp, flat_buffers = lddp.wrap(net, device_ids=[local], buffers=args.ddp_buffers, gradient_as_bucket_view=True,
                                      bucket_cap_mb=args.ddp_bucket_mb, static_graph=bool(args.ddp_static_graph))
    else:
        ddp, flat_buffers = net, None
    trainer = step.LidogTrainer(ddp, num_classes=args.classes, shape=args.shape, buffer_sync=flat_buffers)

    scans = synth.make_batch(args.batch, 1234 + (0 if args.same_data else 1000 * rank), args.shape, args.classes)
    host_pts = [torch.from_numpy(p).pin_memory() for p, _ in scans]
    host_lab = [torch.from_numpy(l).pin_memory() for _, l in scans]
    dev_pts = [p.to(dev) for p in host_pts]
    dev_lab = [l.to(dev) for l in host_lab]
    n_points = sum(p.shape[0] for p in host_pts)
    h2d_bytes = sum(p.numel() * 4 for p in host_pts) + sum(l.numel() * 4 for l in host_lab)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host = {}

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        mecoords.SYNC_WAIT.update(seconds=0.0, count=0)
        marks = []
        gc.collect()
        gc.disable()  # a generation-2 collection inside the loop stalls one rank for tens of ms -- and, through the
        t0 = time.perf_counter()  # SyncBN exchanges, every other rank with it
        e0.record()
        for _ in range(steps):
            fn()
            m = torch.cuda.Event(enable_timing=True)
            m.record()
            marks.append(m)
        e1.record()
        gc.enable()
        host["issue_ms"] = 1e3 * (time.perf_counter() - t0) / steps  # wall time of the host loop, waits included
        host["wait_ms"] = 1e3 * mecoords.SYNC_WAIT["seconds"] / steps  # of which: blocked in the step's one sync
        barrier()
        host["step_ms"] = [round(a.elapsed_time(b), 2) for a, b in zip([e0] + marks[:-1], marks)]  # this rank's steps
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    last = {}

    def resident_step():
        if args.empty_cache:
            torch.cuda.empty_cache()
        last["loss"] = trainer.training_step(dev_pts, dev_lab)

    def e2e_step():
        if args.empty_cache:
            torch.cuda.empty_cache()
        pts = [p.to(dev, non_blocking=True) for p in host_pts]
        lab = [l.to(dev, non_blocking=True) for l in host_lab]
        return float(trainer.training_step(pts, lab).item())  # D2H read of the loss

    if args.ncu:
        resident_step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()
        resident_step()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
        return
    for _ in range(max(args.warmup, 3)):
        resident_step()

    # ---- headline: the UNINSTRUMENTED loop (no per-launch events, no call counting)
    sampler = ClockSampler(local) if rank == 0 else None
    total_ms = timed(resident_step, args.steps)
    host_issue_ms, host_wait_ms = host.get("issue_ms"), host.get("wait_ms")
    step_ms = host.get("step_ms")
    clocks = sampler.stop() if sampler else None
    ms_per_step = total_ms / args.steps
    value = world * args.batch / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:  # before the passes below train the model further
        dump_outputs(args.dump_outputs, net, last["loss"])

    # ---- separate passes (untimed for the headline): launch census, pair census, per-launch kernel times
    cabi.counting(True)
    resident_step()
    torch.cuda.synchronize()
    launches = cabi.kernel_launches()
    cabi.counting(False)
    recs, inst_ms, k_steps = [], 1.0, 1
    # Instrumented pass: every rank runs the same steps (the SyncBN exchanges and the DDP all-reduce need all of them),
    # rank 0 alone wraps its convolution launches in CUDA events -- at N > 1 the roofline is rank 0's kernels inside
    # a data-parallel step, NCCL traffic included.
    prof = rank == 0
    meconv.PROFILE.update(enabled=prof, events=False)
    meconv.PROFILE["records"].clear()
    resident_step()
    torch.cuda.synchronize()
    k_steps = min(args.steps, 4)
    meconv.PROFILE.update(enabled=prof, events=prof)
    meconv.PROFILE["records"].clear()
    inst_ms = timed(resident_step, k_steps)
    recs = list(meconv.PROFILE["records"])
    meconv.PROFILE.update(enabled=False, events=False)

    # roofline of the dominant kernel (tcgen05 gather-GEMM: fwd + dgrad launches), from the instrumented pass
    pk = peaks()
    torch.cuda.synchronize()
    by_kind = {}
    for r in recs:
        k = by_kind.setdefault(r["kernel"], dict(flops=0.0, ms=0.0, n=0))
        k["flops"] += r["flops"]; k["ms"] += r["e0"].elapsed_time(r["e1"]); k["n"] += 1
    roofline = None
    if "k_gemm_tc" in by_kind:
        g = by_kind["k_gemm_tc"]
        ach = g["flops"] / (g["ms"] / 1e3) / 1e12
        traffic, traffic_src = ncu_traffic()
        roofline = {"bound": "tensor", "kernel": "k_gemm2 (tcgen05 gather-GEMM, sparse-conv fwd+dgrad)",
                    "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"],
                    "traffic": traffic,
                    "traffic_note": None if traffic is None else
                    f"dram read+write bytes of ONE launch of the block8 layer shape (ts 1, 96->96, 648k voxels) from "
                    f"profiles/{traffic_src}; its algorithmic bytes are 124 MB fp16 operand + 249 MB fp32 result + "
                    f"70 MB neighbour table; achieved/launches/avg_launch_ms aggregate all launches of a step",
                    "peak_source": pk["source"] + " bf16 sustained (kernel timed inside a long step)",
                    "launches": g["n"], "avg_launch_ms": g["ms"] / g["n"],
                    "share_of_step": g["ms"] / inst_ms,
                    "timing": f"CUDA events around every launch in a separate instrumented pass of {k_steps} steps "
                              f"({inst_ms / k_steps:.2f} ms/step); the headline loop carries no instrumentation",
                    "algorithmic_flops_per_step": g["flops"] / k_steps}
    kernels = {k: {"ms_per_step": v["ms"] / k_steps, "tflops": v["flops"] / (v["ms"] / 1e3) / 1e12 if v["ms"] else None,
                   "launches_per_step": v["n"] / k_steps} for k, v in by_kind.items()}
    conv_ms = sum(v["ms"] for v in by_kind.values()) / k_steps

    # end to end: pinned host buffers -> device each step, loss read back each step
    for _ in range(2):
        e2e_step()
    e2e_ms = timed(e2e_step, args.steps) / args.steps
    e2e = {"value": world * args.batch / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
           "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms}

    if rank == 0:
        sys.stderr.write(f"[bench] {value:.2f} scans/s resident, {e2e['value']:.2f} e2e, {ms_per_step:.1f} ms/step, "
                         f"sparse conv {conv_ms / args.batch:.2f} ms/scan, roofline {roofline}\n")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline(args)
        except Exception as e:  # the baseline is a reported number, never a reason to lose the GPU line
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e!r}"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16 operands / f32 accumulate (tcgen05 kind::f16); f32 elsewhere",
                "data": "synthetic",
                "config": {"workload": f"LiDOG MinkUNet34BEV training step (voxelise + maps + sparse conv fwd/bwd + BEV "
                                       f"projection + cuDNN 2D head + losses + Adam), synthetic {args.shape}-shaped "
                                       f"scans, batch {args.batch}/GPU, {args.classes} classes "
                                       f"(BASELINE {CONFIG_OF_SHAPE[args.shape]})",
                           "points_per_step_per_gpu": n_points, "global_batch": world * args.batch,
                           "parallelism": f"dp{world}" + ((" (DDP gradient all-reduce over NCCL; SyncBN exchange: " +
                                                           ("in-kernel over NVLink peer memory" if mepeer.active()
                                                            else "NCCL all_reduce") + ")") if world > 1 else ""),
                           "nccl_max_ctas": args.nccl_ctas if world > 1 else None,
                           "diagnostic_flags": [f for f, on in (("no_syncbn", args.no_syncbn), ("same_data", args.same_data)) if on],
                           "ddp_bucket_cap_mb": args.ddp_bucket_mb if world > 1 else None,
                           "ddp_buffers": ({"flat": "rank 0's buffers broadcast before every forward as 2 flat tensors "
                                                    "(lidog/ddp.py; same semantics as DDP broadcast_buffers=True)",
                                            "ddp": "DistributedDataParallel(broadcast_buffers=True)",
                                            "off": "not broadcast"}[args.ddp_buffers] if world > 1 else None),
                           "empty_cache_every_step": bool(args.empty_cache),
                           "arena_bytes": int(cabi.lib().lg_arena_bytes()),
                           "l2": "per-step working set (GBs of activations) far exceeds the 126 MB L2; no flush needed",
                           "conv_operands": meconv.CONFIG["tc"], "gather": "cp.async+mbarrier super-tile pipeline, mask-sorted plans",
                           "layer_calls": bool(meconv.CONFIG["layer_calls"]), "epilogue_bn_stats": bool(meconv.CONFIG["epi_stats"]),
                           "fused_bn": bool(menorm.CONFIG["fused"]),
                           "bev_layout": "channels_last" if lbev.CONFIG["channels_last"] else "nchw"},
                # own kernels (liblidog_b200.so) launched inside the timed region: a census step counts them per step
                # (the census is a separate, untimed step: the headline loop carries no counting), per rank
                "e2e": e2e, "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
                "clocks": clocks, "roofline": roofline,
                "sparse_conv_ms_per_scan": conv_ms / args.batch, "kernels": kernels,
                "rank0_step_ms": step_ms,  # per step of the headline loop, CUDA events on rank 0 (diagnostic)
                "host_issue_ms_per_step": host_issue_ms, "host_wait_ms_per_step": host_wait_ms,
                "host_busy_ms_per_step": None if host_issue_ms is None else host_issue_ms - host_wait_ms,
                "host_note": "issue = wall time of the Python loop for one step; wait = the part spent blocked in the "
                             "step's single synchronisation (coordinate-level counts, waiting for the GPU to drain the "
                             "previous step); busy = issue - wait = the CPU work of launching a step",
                "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
