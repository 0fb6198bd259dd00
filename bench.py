#!/usr/bin/env python
"""Benchmark of the view-synthesis loss hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # the sm_100a path
    python bench.py --impl reference --gpus N --steps K ...    # reference algorithm on host cores

One *step* = one pass of the hot path over one synthetic batch: disparity -> depth,
identity pre-pass, warp + SSIM/L1 + per-pixel minimum over every source, smoothness,
forward and backward (gradients to every disparity scale and to the poses).
Metric: warped px-pairs per second (SURVEY.md 8d), whole job over all ranks.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every key.

    python bench.py ... --dump-outputs DIR

also writes what the last timed step computed (losses, the gradients of every leaf, the depth planes) as
DIR/<name>.npy, so that two builds can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

import torch  # noqa: E402

METRIC = "warped px-pairs/s fwd+bwd (photometric loss)"
UNIT = "px-pairs/s"
DEFAULT_WORKLOAD = "kitti_640x192_b12_pm1"   # BASELINE.json configs[1]
_REAL_STDOUT = 1


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-full-step", action="store_true",
                    help="skip the full-training-step sub-record (BASELINE.json configs[4])")
    ap.add_argument("--with-pose", action="store_true",
                    help="include the pose assembly (axis-angle/translation -> T, SURVEY 8f-2) in the timed step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload in FULL_STEP):
        ap.error("--dump-outputs covers the fused loss path (--impl ours, a loss workload)")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def collect_outputs(losses, leaves, outputs):
    """What a caller of loss_step + backward receives from one step: the losses, the gradient of every leaf and
    the depth planes loss_step stores in ``outputs``; copied to the host as float32 numpy arrays."""
    def name(k):
        return "_".join(str(p) for p in k) if isinstance(k, tuple) else str(k)

    arrays = {name(k).replace("/", "_"): v for k, v in losses.items()}
    arrays.update({"grad_" + name(k): p.grad for k, p in leaves.items()})
    arrays.update({name(k): v for k, v in outputs.items() if isinstance(k, tuple) and k[0] == "depth"})
    return {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}


def write_outputs(directory, arrays):
    """Save ``arrays`` as ``directory/<name>.npy``.  Past DUMP_LIMIT_BYTES in all, every array keeps the same share of
    its elements, picked by a fixed seed (flat indices, ascending), so that two runs keep the same elements."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    room = DUMP_LIMIT_BYTES - 1024 * len(arrays)          # the .npy headers
    keep = min(1.0, room / total) if total else 1.0
    for k, a in sorted(arrays.items()):
        if keep < 1.0 and a.size > 1:
            idx = np.sort(np.random.default_rng(0).choice(a.size, max(1, int(a.size * keep)), replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(directory, k + ".npy"), a)


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0 = index, [], None, 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [c.strip() for c in line.split(",")])

    def mark(self):
        """Only samples that arrive after this call count (the GPU is under load from here on)."""
        self.t0 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7 or r[0] < self.t0:
                continue
            r = r[1:]
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload(name):
    from baseboostdepth_b200.synthetic import WORKLOADS
    B, H, W, baselines, trimin, decomp = WORKLOADS[name]
    return dict(batch=B, height=H, width=W, baselines=list(baselines), trimin=trimin, decomp=decomp)


def make_opt(cfg):
    from types import SimpleNamespace
    return SimpleNamespace(height=cfg["height"], width=cfg["width"], scales=[0, 1, 2, 3], min_depth=0.1,
                           max_depth=100.0, disparity_smoothness=1e-3, no_ssim=False, trimin=cfg["trimin"],
                           decomp=cfg["decomp"], pose_error=5.5, SQL=False, batch_size=cfg["batch"])


# ----------------------------------------------------------------------------------------------
def cpu_reference_run(cfg, steps, warmup, sample_batch=None):
    """The reference algorithm (oracle port, plain PyTorch ops) on the host cores.

    Returns (px-pairs/s, seconds per step, sample description, threads)."""
    from baseboostdepth_b200.plan import build_plan
    from baseboostdepth_b200.synthetic import make_batch, make_noise, px_pairs
    from oracle import loss_path as O

    c = dict(cfg)
    if sample_batch is not None and sample_batch < c["batch"]:
        c["baselines"] = c["baselines"][:sample_batch]
        c["batch"] = sample_batch
    opt = make_opt(c)
    inputs, outputs, params = make_batch(seed=1234, device="cpu", pose_error=5.5, **c)
    plan = build_plan(inputs["ordering"], trimin=c["trimin"], decomp=c["decomp"])
    noise = make_noise(plan, c["height"], c["width"])
    pairs = px_pairs(plan, c["height"], c["width"], 4)
    # use every host thread unless that is slower than one (oversubscribed / quota-limited hosts)
    probe = {}
    for n in sorted({os.cpu_count() or 1, 1}, reverse=True):
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        with torch.no_grad():
            O.run(inputs, dict(outputs), opt, noise, num_scales=4)
        probe[n] = time.perf_counter() - t0
    threads = min(probe, key=probe.get)
    torch.set_num_threads(threads)
    times = []
    for it in range(warmup + steps):
        for p in params.values():
            p.grad = None
        fresh = {k: v for k, v in outputs.items() if k[0] in ("disp", "cam_T_cam", "cam_T_cam_error")}
        # poses must be rebuilt from their leaves each step (the graph is consumed by backward)
        from baseboostdepth_b200.geometry import transformation_from_parameters
        for k in list(fresh):
            if k[0] == "cam_T_cam" and ("axisangle", k[2]) in params:
                fresh[k] = transformation_from_parameters(params[("axisangle", k[2])], params[("translation", k[2])],
                                                          invert=(k[2] < 0))
        t0 = time.perf_counter()
        out, _ = O.run(inputs, fresh, opt, noise, num_scales=4)
        out["loss"].backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    sample = (f"{c['batch']} of {cfg['batch']} samples of the workload, all scales and sources, "
              f"{steps} timed steps after {warmup} warm-up, {threads} threads")
    cpu_reference_run.last_probe = {str(k): v for k, v in probe.items()}   # forward-only seconds per thread count
    return pairs / sec, sec, sample, threads


def eager_cuda_ms(cfg, dev, steps=5):
    """Baseline leg: the oracle port (reference algorithm, plain ATen ops) evaluated eagerly on the GPU."""
    from baseboostdepth_b200.plan import build_plan
    from baseboostdepth_b200.synthetic import make_batch, make_noise
    from oracle import loss_path as O
    inputs, outputs, params = make_batch(seed=1234, device=dev, pose_error=5.5, **cfg)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in outputs.items()
              if k[0] in ("disp", "cam_T_cam") and v.numel()}
    plan = build_plan(inputs["ordering"], trimin=cfg["trimin"], decomp=cfg["decomp"])
    noise = {g: n.to(dev) for g, n in make_noise(plan, cfg["height"], cfg["width"]).items()}
    opt = make_opt(cfg)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for it in range(steps + 2):
        for p in leaves.values():
            p.grad = None
        outs = {k: leaves.get(k, v) for k, v in outputs.items() if k[0] in ("disp", "cam_T_cam", "cam_T_cam_error")}
        ev0.record()
        out, _ = O.run(inputs, outs, opt, noise, num_scales=4)
        out["loss"].backward()
        ev1.record()
        torch.cuda.synchronize()
        if it >= 2:
            ms.append(ev0.elapsed_time(ev1))
    return sum(ms) / len(ms)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = workload(args.workload)
    # the metric's own configuration: the full batch, all scales and sources, the K / W the caller asked for
    # (~0.5-3 s per step on the box's host cores depending on the workload)
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    value, sec, sample, threads = cpu_reference_run(cfg, steps, warmup, sample_batch=None)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "batch_per_gpu": cfg["batch"], "height": cfg["height"],
                       "width": cfg["width"], "scales": 4, "device": "host CPU", "threads": threads,
                       "host_cores": os.cpu_count(),
                       "thread_probe_forward_s": getattr(cpu_reference_run, "last_probe", None),
                       "note": "oracle port of the reference's PyTorch loss path (reference is Python; "
                               "/root/reference cannot travel to the GPU box); full batch, same workload as the GPU arm"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ----------------------------------------------------------------------------------------------
def run_ours(args):
    from baseboostdepth_b200 import _lib
    from baseboostdepth_b200.geometry import transformation_from_parameters
    from baseboostdepth_b200.synthetic import algorithmic_bytes, make_batch, make_noise, px_pairs
    from baseboostdepth_b200.trainer import loss_step, plan_for

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from baseboostdepth_b200.staging import bind_to_gpu_numa
    try:   # NVML indexes physical devices; CUDA_VISIBLE_DEVICES may remap (or hold UUIDs)
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        numa = bind_to_gpu_numa(int(vis.split(",")[local]) if vis else local)
    except (ValueError, IndexError):
        numa = "not bound (CUDA_VISIBLE_DEVICES is not a list of indices)" 
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()           # nvidia-smi needs ~0.5 s to come up; samples are filtered by mark()
    cfg = workload(args.workload)
    opt = make_opt(cfg)
    H, W = cfg["height"], cfg["width"]
    inputs, outputs, params = make_batch(seed=1234 + rank, device=dev, pose_error=5.5, **cfg)
    plan = plan_for(inputs["ordering"], cfg["trimin"], cfg["decomp"],
                    inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
    noise = {g: n.to(dev) for g, n in make_noise(plan, H, W, seed=4321 + rank).items()}
    pairs = px_pairs(plan, H, W, 4)
    abytes = algorithmic_bytes(plan, H, W, [0, 1, 2, 3])
    be = _lib.cuda_backend()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # The path's inputs are disparities and camera motions T (SURVEY.md 8a/b: gradients are required for
    # depth/disp and T); the motions become leaves here.  Assembling T from axis-angle/translation is
    # the reference's predict_poses, a "next" row (SURVEY.md 8f-2), outside the timed path.
    leaves = {k: v for k, v in params.items() if k[0] == "disp"}
    pose_params = {}
    if args.with_pose:
        # --with-pose: the leaves are the pose network's outputs (axis-angle, translation); every step assembles the
        # camera motions with the library's pose kernel (layers.transformation_from_parameters: one launch forward,
        # one backward per frame instead of the reference's ~40 tiny tensor kernels, layers.py:25-100)
        from baseboostdepth_b200.layers import transformation_from_parameters as pose_op
        for k, v in params.items():
            if k[0] in ("axisangle", "translation"):
                pose_params[k] = v.detach().clone().requires_grad_(True)
                leaves[k] = pose_params[k]
    else:
        for k in list(outputs):
            if k[0] == "cam_T_cam" and outputs[k].numel():
                outputs[k] = outputs[k].detach().clone().requires_grad_(True)
                leaves[k] = outputs[k]

    def rebuild_poses():
        if not args.with_pose:
            return
        for f in plan.frames:
            if f == "s":
                continue
            outputs[("cam_T_cam", 0, f)] = pose_op(pose_params[("axisangle", f)], pose_params[("translation", f)], invert=(f < 0))

    timers = {}

    def step():
        rebuild_poses()
        # noise=None: the tie-break noise is drawn on the device inside the step, one torch.randn per
        # baseline group, exactly like compute_losses does (trainer.py:518-523)
        losses = loss_step(inputs, outputs, opt, plan, noise=None, num_scales=4, timers=timers)
        losses["loss"].backward()
        return losses

    # ---- device-resident timing ------------------------------------------------------------
    torch.manual_seed(4321 + rank)   # the noise drawn inside the steps: the same from run to run
    sampler.mark()                # clock samples count from the warm-up to the end of the e2e loop
    for _ in range(max(3, args.warmup)):
        for p in leaves.values():
            p.grad = None
        step()
    barrier()
    be.launches = 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ev = []
    barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        for p in leaves.values():
            p.grad = None
        if not os.environ.get("BBD_BENCH_NO_FLUSH"): flush.zero_()
        timers.clear()
        ev[i][0].record()
        last = step()
        ev[i][1].record()
        kernel_ev.append(timers.get("reproj_fused"))
    barrier()
    wall = time.perf_counter() - wall0
    dump = collect_outputs(last, leaves, outputs) if args.dump_outputs and rank == 0 else None
    launches = be.launches
    step_ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
    kern_ms = sum(a.elapsed_time(b) for a, b in kernel_ev if a is not None) / max(1, len(kernel_ev))
    kernel_name = timers.get("reproj_kernel_name", "bbd::reproj_kernel")

    # ---- per-kernel durations of the rest of the step: the same eager step with every launch of ours bracketed
    # by CUDA events on its own stream (L2 flushed before each step), mean over a few steps
    per_call = {}
    for i in range(min(10, args.steps)):
        for p in leaves.values():
            p.grad = None
        if not os.environ.get("BBD_BENCH_NO_FLUSH"): flush.zero_()
        timers.clear()
        step()
        torch.cuda.synchronize()
        for k, v in timers.items():
            if isinstance(v, tuple):
                per_call.setdefault(k, []).append(v[0].elapsed_time(v[1]))
    per_call = {k: sum(v) / len(v) for k, v in per_call.items()}

    # ---- the same step captured once in a CUDA graph and replayed (no Python / launch overhead) ----
    graph_ms = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                # fresh leaves: their gradient-accumulation nodes must not belong to the legacy default stream
                # the eager loop above ran on (autograd would make that stream wait for the capturing one, which
                # invalidates the capture)
                for k in list(leaves):
                    leaves[k] = leaves[k].detach().clone().requires_grad_(True)
                    if k in pose_params:
                        pose_params[k] = leaves[k]
                    else:                                    # ("disp", s) and ("cam_T_cam", 0, f) are outputs entries
                        outputs[k] = leaves[k]
                for _ in range(3):
                    for p in leaves.values():
                        p.grad = None
                    step()
            torch.cuda.current_stream().wait_stream(side)
            for p in leaves.values():
                p.grad = None
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                static_losses = step()
            gev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            barrier()
            for i in range(args.steps):
                if not os.environ.get("BBD_BENCH_NO_FLUSH"): flush.zero_()
                gev[i][0].record()
                g.replay()
                gev[i][1].record()
            barrier()
            graph_ms = sum(a.elapsed_time(b) for a, b in gev) / args.steps
            if dump is not None:    # the replayed step is the headline: its last replay is what gets written
                dump = collect_outputs(static_losses, leaves, outputs)
        except Exception as exc:  # noqa: BLE001
            graph_ms = None
            print(f"graph capture failed: {type(exc).__name__}: {exc}", file=sys.stderr)
            if os.environ.get("BBD_BENCH_DEBUG"):
                import traceback
                traceback.print_exc()
    if dump is not None:
        write_outputs(args.dump_outputs, dump)

    # ---- end to end: pinned host batch -> H2D -> fused loss fwd+bwd -> D2H loss ---------------
    # Every step uploads its whole batch (images, pyramid, K, stereo_T, disparities, camera motions)
    # from pinned host memory; BatchStager moves it as one DMA on a side stream, double-buffered,
    # so step i+1's upload overlaps step i's kernels.  The loss value is read back every step.
    e2e_ms, h2d, e2e8_ms, h2d8, e2e_graphed, h2d_gbs = None, 0, None, 0, False, 0.0
    if not args.no_e2e:
        from baseboostdepth_b200.staging import BatchStager

        def is_frame(k):      # colour frames and the colour pyramid: 8-bit images when they leave the decoder
            return isinstance(k, tuple) and k[0] == "color"

        def e2e_measure(frames_8bit):
            # What a data loader hands over crosses PCIe: the colour frames (and K / inv_K / stereo_T).  The colour
            # pyramid levels 1..3 are derived on the device from the uploaded frame (mono_dataset.py:187-204 builds
            # them on the host by resizing), disparities and camera motions are born on the device (network outputs).
            template = {}
            for k, v in inputs.items():
                if torch.is_tensor(v):
                    if is_frame(k) and k[2] != 0:
                        continue                                 # pyramid level: derived on the device
                    if frames_8bit and is_frame(k):
                        v = (v * 255).round().to(torch.uint8)
                    template[("in",) + (k if isinstance(k, tuple) else (k,))] = v
            stager = BatchStager(template, dev)

            import torch.nn.functional as F
            dev_leaves = {k: v.detach().clone() for k, v in leaves.items() if k[0] in ("disp", "cam_T_cam")}

            def make_io(v):
                gin = {"ordering": inputs["ordering"]}
                gout, lv = {}, {}
                for k, t in v.items():
                    gin[k[1] if len(k) == 2 else k[1:]] = t
                for k, t in dev_leaves.items():
                    gout[k] = lv[k] = t.detach().requires_grad_(True)
                for k in outputs:
                    if k[0] == "cam_T_cam" and k not in gout:
                        gout[k] = outputs[k]
                return gin, gout, lv

            def derive_pyramid(gin):
                c0 = gin[("color", 0, 0)]
                for s_ in (1, 2, 3):
                    gin[("color", 0, s_)] = F.avg_pool2d(c0, 2 ** s_)
                return gin

            def with_error_poses(gout):
                if cfg["decomp"]:
                    for k in [k for k in gout if k[0] == "cam_T_cam"]:
                        te = gout[k].detach().clone()
                        te[:, :3, 3:] /= 5.5
                        gout[("cam_T_cam_error", 0, k[2])] = te
                return gout

            graphed = None
            if not args.no_graph:
                try:
                    from baseboostdepth_b200.graphed import GraphedLossStep
                    graphed = GraphedLossStep(stager, make_io, opt, plan, num_scales=4, prepare=with_error_poses,
                                              prepare_inputs=derive_pyramid)
                except Exception as exc:  # noqa: BLE001
                    print(f"graphed e2e unavailable: {type(exc).__name__}: {exc}", file=sys.stderr)

            def consume(slot):
                gin, gout, _ = make_io(stager.views(slot))
                losses = loss_step(derive_pyramid(gin), with_error_poses(gout), opt, plan, noise=None, num_scales=4)
                losses["loss"].backward()
                stager.release(slot)
                return losses["loss"].detach()

            def e2e_run(n):
                pending = stager.upload_async()
                total = 0.0
                for i in range(n):
                    slot = pending
                    if i + 1 < n:
                        pending = stager.upload_async()      # next batch crosses PCIe during this step
                    if graphed is not None:
                        graphed.launch(slot)                 # one cudaGraphLaunch
                        v = graphed.collect()                # device -> host read of the previous step's loss
                        total += v if v is not None else 0.0
                    else:
                        total += float(consume(slot))        # device -> host read of the step's result
                if graphed is not None:
                    total += graphed.collect(final=True)
                return total

            e2e_run(3)
            barrier()
            n_e2e = args.steps
            runs = []
            for _ in range(3):                       # three timed loops, the median is reported
                if not os.environ.get("BBD_BENCH_NO_FLUSH"): flush.zero_()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e2e_run(n_e2e)
                torch.cuda.synchronize()
                runs.append((time.perf_counter() - t0) / n_e2e * 1e3)
            barrier()
            return sorted(runs)[1], stager.nbytes, graphed is not None

        # host -> device ceiling of this rank while every rank uploads at once (what bounds the fp32 variant)
        probe_h = torch.empty(128 << 20, dtype=torch.uint8).pin_memory()
        probe_d = torch.empty(128 << 20, dtype=torch.uint8, device=dev)
        probe_d.copy_(probe_h, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(8):
            probe_d.copy_(probe_h, non_blocking=True)
        torch.cuda.synchronize()
        h2d_gbs = 8 * probe_h.numel() / (time.perf_counter() - t0) / 1e9
        del probe_h, probe_d
        e2e_ms, h2d, e2e_graphed = e2e_measure(False)   # fp32 host tensors, as the reference's loader hands them over
        e2e8_ms, h2d8, _ = e2e_measure(True)            # frames kept 8-bit on the host, expanded on the device

    # keep the GPU busy long enough for a handful of 100 ms clock samples, then stop the sampler
    t_busy = time.perf_counter()
    while rank == 0 and time.perf_counter() - t_busy < 0.6:
        step()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None

    # ---- max over ranks ------------------------------------------------------------------------
    vals = torch.tensor([step_ms, kern_ms, e2e_ms or 0.0, wall * 1e3 / args.steps, graph_ms or 0.0, e2e8_ms or 0.0,
                         -h2d_gbs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    step_ms, kern_ms, e2e_ms_max, wall_ms, graph_ms_max, e2e8_ms_max, neg_gbs = (float(v) for v in vals.cpu())
    h2d_gbs_min = -neg_gbs   # slowest rank's host->device bandwidth with all ranks copying

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (
            6650.0, "fallback (B200_PROFILING.md)")
        achieved = abytes["reproj"] / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else None
        traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of the same kernel, one ncu --set full capture
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload)
        except (OSError, ValueError):
            pass
        other_bytes = {"ident_forward": abytes["identity"], "smooth_fused": abytes["smooth"],
                       "disp_to_depth_forward": abytes["d2d_forward"], "disp_to_depth_backward": abytes["d2d_backward"],
                       "reproj_finalize": None}
        others = [{"call": "bbd_" + k, "us": per_call[k] * 1e3, "algorithmic_bytes": other_bytes.get(k),
                   "frac": (other_bytes[k] / (per_call[k] * 1e-3) / 1e9 / peak) if other_bytes.get(k) else None}
                  for k in ("ident_forward", "smooth_fused", "disp_to_depth_forward", "reproj_finalize",
                            "disp_to_depth_backward") if k in per_call]
        # headline: the step as the public API runs it in a training loop -- captured once, replayed as a
        # CUDA graph (graphed.GraphedLossStep does the same per staging slot); the eagerly launched step
        # (Python + 14 launches + 3 tensor ops per step) is reported beside it
        eager_ms = step_ms
        if graph_ms is not None and graph_ms_max > 0:
            step_ms = graph_ms_max
        line = {
            "metric": METRIC, "value": pairs * world / (step_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "batch_per_gpu": cfg["batch"], "height": H, "width": W,
                       "scales": 4, "px_pairs_per_step_per_gpu": pairs, "sharding": f"batch x{world}, no data-path collective",
                       "l2": "flushed between steps (256 MiB memset, outside the per-step events)",
                       "timing": "CUDA events per step on the launch stream, mean over steps, max over ranks; "
                                 + ("the step is captured once and replayed as a CUDA graph" if step_ms != eager_ms
                                    else "eager launches"),
                       "with_pose": bool(args.with_pose), "eager_ms_per_step": eager_ms, "eager_wall_ms_per_step_incl_flush": wall_ms,
                       "cuda_graph_replay_ms_per_step": graph_ms_max if graph_ms is not None else None},
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "peak_source": peak_src, "kernel_ms": kern_ms,
                         "algorithmic_bytes_per_launch": abytes["reproj"],
                         "step_algorithmic_bytes": abytes["total"],
                         "step_frac": abytes["total"] / (step_ms * 1e-3) / 1e9 / peak,
                         "kernel_share_of_eager_step": kern_ms / eager_ms,
                         "frac_vs_spec_sheet_8000_GBs": (achieved / 8000.0) if achieved else None,
                         "others": others,
                         "others_note": "C-ABI calls of the same step besides the fused kernel, each bracketed by CUDA events "
                                        "on its own stream in an eager pass (several run concurrently on helper streams, so "
                                        "their sum exceeds their share of the step); bytes per SURVEY 8(d)"},
            "clocks": clocks, "gpu_launches": launches,
        }
        if e2e_ms is not None:
            line["e2e"] = {"value": pairs * world / (e2e_ms_max * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_max,
                           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                           "h2d_gbs_per_gpu_all_ranks_copying": h2d_gbs_min,
                           "h2d_floor_ms_per_step": (h2d / (h2d_gbs_min * 1e9) * 1e3) if h2d_gbs_min > 0 else None,
                           "uploaded": "what a loader provides: colour frames of every source + K, inv_K, stereo_T; the colour "
                                       "pyramid levels 1-3 are derived on the device, disparities and camera motions are "
                                       "device-resident network outputs",
                           "how": "loss_step + backward on a batch uploaded from a pinned host arena each step "
                                  "(single DMA, double-buffered on a side stream), "
                                  + ("the step replayed as a CUDA graph per staging slot (graphed.GraphedLossStep), every "
                                     "step's loss read back one step behind; " if e2e_graphed else "loss read back each step; ")
                                  + "wall clock over the loop, median of 3 loops; working set 2 x batch > L2",
                           "host_affinity": numa,
                           "frames_8bit": {"value": pairs * world / (e2e8_ms_max * 1e-3), "ms_per_step": e2e8_ms_max,
                                           "h2d_bytes_per_step": h2d8,
                                           "how": "same loop with the colour frames staged as the decoder's "
                                                  "8-bit samples and expanded on the device (bbd_u8_to_f32 == ToTensor, "
                                                  "bit-identical) -- the upload is PCIe-bound at N > 1 otherwise"}}
        if not args.no_cpu_baseline and world == 1:
            v, sec, sample, threads = cpu_reference_run(cfg, steps=3, warmup=1, sample_batch=None)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                                    "s_per_step": sec,
                                    "thread_probe_forward_s": getattr(cpu_reference_run, "last_probe", None)}
            # context only: the same oracle code run eagerly on this GPU (what the reference's ATen path costs)
            try:
                line["cpu_baseline"]["same_code_eager_cuda_ms_per_step"] = eager_cuda_ms(cfg, dev)
            except Exception as exc:  # noqa: BLE001
                line["cpu_baseline"]["same_code_eager_cuda_ms_per_step"] = f"failed: {type(exc).__name__}"
    # ---- BASELINE.json configs[4] beside the headline: the full training step on the same N GPUs, with its
    # NCCL leg (gradient all-reduce of the surrounding networks; the loss path itself has no collective)
    full = None
    if not args.no_full_step and args.workload == DEFAULT_WORKLOAD:
        try:
            full = full_step_record(args, dev, world, rank, local, cfg["batch"], H, W, steps=args.steps,
                                    context_legs=False)
        except Exception as exc:  # noqa: BLE001
            full = {"unavailable": f"{type(exc).__name__}: {exc}"}
    if rank == 0:
        if full is not None:
            line["full_step"] = {k: full[k] for k in ("metric", "value", "unit", "ms_per_step", "config", "e2e", "unavailable")
                                 if k in full}
        emit(line)
    if world > 1:
        dist.destroy_process_group()

# ----------------------------------------------------------------------------------------------
FULL_STEP = {"full_step_640x192_b12": (12, 192, 640), "full_step_1024x320_b8": (8, 320, 1024)}


def full_step_record(args, dev, world, rank, local, B, H, W, steps, context_legs=True):
    """BASELINE.json configs[4] measured in this process (process group, if any, already initialised):
    networks + fused loss + Adam, batch-sharded, DDP all-reduce of the network gradients over NCCL.  Returns
    (record, sampler clocks or None); rank 0's record is meaningful."""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import full_step as FS
    from baseboostdepth_b200 import _lib
    if world > 1:
        import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    be = _lib.cuda_backend()
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v)
            for k, v in FS.make_inputs(B, H, W, "cpu", seed=1234 + rank).items()}
    inputs = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))

    def timed(trainer, n, warmup, upload=False, no_sync=False):
        import contextlib
        ctx = trainer.ddp.no_sync if (no_sync and trainer.ddp is not None) else contextlib.nullcontext
        with ctx():
            for _ in range(warmup):
                trainer.step(inputs)
            barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            ev0.record()
            last = None
            for _ in range(n):
                if upload:
                    batch = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in host.items()}
                    last = float(trainer.step(batch)["loss"])
                else:
                    last = trainer.step(inputs)["loss"]
            ev1.record()
            barrier()
        wall = (time.perf_counter() - t0) / n * 1e3
        ms = ev0.elapsed_time(ev1) / n
        t = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), float(last)

    warm = max(3, args.warmup)
    torch.manual_seed(1)
    fused = FS.StepTrainer(B, H, W, dev, loss="fused", ddp=world > 1, local_rank=local)
    timed(fused, 2, warm)
    be.launches = 0
    runs = [timed(fused, steps, 0) for _ in range(3)]        # eager PyTorch launching ~1,600 kernels per step is
    launches = be.launches // 3                               # jittery: the median of three timed loops is reported
    ms, _, loss = sorted(runs)[1]
    nosync_ms = sorted(timed(fused, steps, 1, no_sync=True)[0] for _ in range(3))[1] if world > 1 else None
    _, e2e_wall, _ = timed(fused, steps, 2, upload=True)
    legs = {}
    for name in (("none", "eager") if context_legs else ("none",)):   # same networks and optimiser, other loss
        torch.manual_seed(1)
        other = FS.StepTrainer(B, H, W, dev, loss=name, ddp=world > 1, local_rank=local)
        legs[name] = sorted(timed(other, steps, 3 if i == 0 else 0)[0] for i in range(3))[1]
        del other
        torch.cuda.empty_cache()
    n_params = fused.n_params
    del fused
    torch.cuda.empty_cache()
    rec = {"metric": "training examples/s (full step: networks + fused view-synthesis loss + Adam)",
           "value": B * world / (ms * 1e-3), "unit": "examples/s", "n_gpus": world, "steps": steps,
           "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"full_step_{W}x{H}_b{B}", "batch_per_gpu": B, "height": H, "width": W, "scales": 4,
                      "frames": [0, -1, 1], "network_parameters": n_params,
                      "networks": "ResNet-18 encoder + skip decoder + 6-channel ResNet-18 pose encoder + pose head, "
                                  "random init, plain torch/cuDNN fp32 (not the product)",
                      "sharding": f"batch x{world}; DistributedDataParallel all-reduce of the network gradients "
                                  f"({n_params * 4 / 1e6:.0f} MB fp32) over NCCL" if world > 1 else "single GPU",
                      "l2": "working set (activations of a 12-sample ResNet step) far exceeds the 126 MB L2",
                      "timing": "CUDA events around K steps, max over ranks, median of 3 such loops",
                      "ms_per_step_all_loops": [r[0] for r in runs],
                      "ms_per_step_networks_only": legs["none"],
                      "ms_per_step_without_gradient_allreduce": nosync_ms,
                      "exposed_allreduce_ms": (ms - nosync_ms) if nosync_ms is not None else None,
                      "ms_per_step_with_stock_pytorch_loss": legs.get("eager"),
                      "loss_share_ms_fused": ms - legs["none"],
                      "loss_share_ms_stock": (legs["eager"] - legs["none"]) if "eager" in legs else None,
                      "final_loss": loss},
           "gpu_launches": launches,
           "e2e": {"value": B * world / (e2e_wall * 1e-3), "unit": "examples/s", "ms_per_step": e2e_wall,
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                   "how": "batch uploaded from pinned host memory every step, loss read back every step; wall clock"}}
    return rec


def run_full_step(args):
    """BASELINE.json configs[4] as the headline of this invocation (``--workload full_step_...``)."""
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    B, H, W = FULL_STEP[args.workload]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    sampler.mark()
    rec = full_step_record(args, dev, world, rank, local, B, H, W, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        rec["clocks"] = clocks
        emit(rec)
    if world > 1:
        dist.destroy_process_group()


def emit(line):
    """The one JSON line, on the process's real stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def main():
    # Libraries may print on stdout (NCCL's version banner does when NCCL_DEBUG is set on the box);
    # the contract is ONE JSON line there, so everything else is routed to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.workload in FULL_STEP:
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                emit({"impl": "reference", "unavailable": "the full-step workload has no CPU reference leg; "
                      "its stock-PyTorch leg is config.ms_per_step_with_stock_pytorch_loss"})
        else:
            run_full_step(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
