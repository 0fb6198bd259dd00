"""Cost of the colour-frame gradients of the fused loss: one JSON line.

    python scripts/frame_grad_bench.py [--steps 50] [--warmup 5] [--out FILE]

For config 1 (kitti_640x192_b12_pm1) and trimin_decomp_640x192_b12 of synthetic.WORKLOADS it times, like
bench.py (warm-up, CUDA events around each step, a 256 MiB memset between steps, median over the steps):
  (a) the fused step (forward + backward) with frames not requiring grad,
  (b) the same step with the target, every source stack and every pyramid level requiring grad,
  (c) the oracle's ATen path (oracle/loss_path.py) on the same GPU with frames requiring grad.
Then a separate torch.profiler run of (b) gives the time of each new kernel; with the bytes each must move at
least (formulas in kernel_bytes) that gives the achieved bandwidth and its share of 7.7 TB/s HBM.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

from baseboostdepth_b200 import _lib  # noqa: E402
from baseboostdepth_b200.synthetic import WORKLOADS, make_batch, make_noise  # noqa: E402
from baseboostdepth_b200.trainer import loss_step, plan_for  # noqa: E402
from oracle import loss_path as O  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
NEW_KERNELS = ("frame_grad_coef_kernel", "frame_grad_pred_kernel", "frame_grad_stack_kernel", "gs_segment_kernel",
               "smooth_image_grad_kernel")


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def kernel_bytes(plan, B, H, W, S, rows):
    """Least traffic of each new kernel (fp32 = 4 bytes, winner = 1 byte, keys / order / segments = 4 bytes)."""
    HW, R = H * W, plan.max_rep
    px = S * B * HW
    return {
        # reads winner, depth, target, one 3-channel candidate value per pixel; writes 18 coefficients
        "frame_grad_coef_kernel": px * (1 + 4 + 12 + 12) + px * 18 * 4,
        # reads the coefficients, winners, depth, candidate values; writes g_pred, keys, target / identity gradients
        "frame_grad_pred_kernel": px * (18 * 4 + 1 + 4 + 12) + px * R * (12 + 4) + B * HW * 12 * (1 + int(plan.hdr[:, 1].max())),
        # reads seg_start, order, g_pred of every entry, depth; writes every stack row
        "gs_segment_kernel": px * R * 4 + rows * HW * 4,
        "frame_grad_stack_kernel": rows * HW * 4 + px * R * (4 + 12 + 4) + rows * 3 * HW * 4,
        # reads disparity and image, writes the image gradient (all levels; level s is 4^-s of level 0)
        "smooth_image_grad_kernel": sum(B * (HW >> (2 * s)) * (4 + 12 + 12) for s in range(S)),
    }


def run_workload(name, steps, warmup):
    dev = torch.device("cuda:0")
    batch, H, W, baselines, trimin, decomp = WORKLOADS[name]
    scales = [0, 1, 2, 3]
    opt = O.default_opt(height=H, width=W, trimin=trimin, decomp=decomp, pose_error=5.5, scales=scales, batch_size=batch)
    cfg = dict(batch=batch, height=H, width=W, baselines=list(baselines), trimin=trimin, decomp=decomp)
    inputs, outputs, params = make_batch(seed=1234, device=dev, scales=scales, **cfg)
    plan = plan_for(inputs["ordering"], trimin, decomp,
                    inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
    leaves = {k: v for k, v in params.items() if k[0] == "disp"}
    for k in list(outputs):
        if k[0] == "cam_T_cam" and outputs[k].numel():
            outputs[k] = outputs[k].detach().clone().requires_grad_(True)
            leaves[k] = outputs[k]
    colour = [k for k in inputs if isinstance(k, tuple) and k[0] == "color"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    noise = {g: n.to(dev) * 1e-5 for g, n in make_noise(plan, H, W, seed=4321).items()}

    def fused_step():
        loss_step(inputs, outputs, opt, plan, noise=None, num_scales=4)["loss"].backward()

    def oracle_step():
        out = {k: v for k, v in outputs.items() if k[0] in ("cam_T_cam", "cam_T_cam_error", "disp")}
        O.run(inputs, out, opt, noise, num_scales=4)[0]["loss"].backward()

    def timed(fn, frames_grad, n_steps):
        for k in colour:
            inputs[k] = inputs[k].detach().requires_grad_(frames_grad)
        torch.manual_seed(4321)
        for _ in range(warmup):
            fn()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        for i in range(n_steps):
            for t in list(leaves.values()) + [inputs[k] for k in colour]:
                t.grad = None
            flush.zero_()
            ev[i][0].record()
            fn()
            ev[i][1].record()
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ev)
        return {"median_ms": ms[len(ms) // 2], "min_ms": ms[0], "max_ms": ms[-1], "steps": n_steps}

    res = {"workload": name, "batch": batch, "height": H, "width": W, "max_rep": plan.max_rep,
           "a_fused_no_frame_grad": timed(fused_step, False, steps),
           "b_fused_frame_grad": timed(fused_step, True, steps),
           "c_oracle_aten_frame_grad": timed(oracle_step, True, steps)}
    res["b_minus_a_ms"] = res["b_fused_frame_grad"]["median_ms"] - res["a_fused_no_frame_grad"]["median_ms"]

    # per-kernel times of the new kernels (profiler on, in a run of its own)
    for k in colour:
        inputs[k] = inputs[k].detach().requires_grad_(True)
    n_prof = 5
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            for t in list(leaves.values()) + [inputs[k] for k in colour]:
                t.grad = None
            fused_step()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        for kn in NEW_KERNELS:
            if kn in e.key:
                t_us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                per[kn] = per.get(kn, 0.0) + t_us / n_prof
    rows = sum(inputs[("color", f, 0)].shape[0] for f in plan.frames)
    nbytes = kernel_bytes(plan, batch, H, W, 4, rows)
    res["new_kernels"] = {
        kn: {"us_per_step": per.get(kn), "algorithmic_bytes": nbytes[kn],
             "achieved_TBps": (nbytes[kn] / (per[kn] * 1e-6) / 1e12) if per.get(kn) else None,
             "share_of_hbm_peak": (nbytes[kn] / (per[kn] * 1e-6) / HBM_BYTES_PER_S) if per.get(kn) else None}
        for kn in NEW_KERNELS}
    res["scratch_bytes_per_step"] = {
        "coef": 4 * 4 * batch * 18 * H * W, "g_pred": 4 * 4 * batch * plan.max_rep * 3 * H * W,
        "keys_and_sorted_keys_and_int32_order": 3 * 4 * 4 * batch * plan.max_rep * H * W,
        "torch_sort_int64_indices": 8 * 4 * batch * plan.max_rep * H * W}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frame_grad_bench.py needs a CUDA device")
    _lib.cuda_backend()
    result = {"card": card(), "method": "CUDA events per step, 256 MiB memset between steps, median",
              "workloads": [run_workload(n, args.steps, args.warmup)
                            for n in ("kitti_640x192_b12_pm1", "trimin_decomp_640x192_b12")]}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
