"""Run the fused path (CUDA library or the CPU emulation harness) on a trainer-style batch."""
from __future__ import annotations

import os
import subprocess
import tempfile

import torch

from baseboostdepth_b200 import _lib
from baseboostdepth_b200.trainer import loss_step, materialise_warps, plan_for

EMU_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
_EMU = None


def emu_backend(flags: str = None) -> _lib.Backend:
    """Compile (if stale) and load tests/emu/libbbd_emu*.so -- the kernels' phase code run on the CPU.
    ``flags`` (or $BBD_EMU_FLAGS): extra -D options selecting a kernel variant, built into its own file.
    Built next to the sources, or in the temporary directory when the tree is read-only."""
    global _EMU
    flags = os.environ.get("BBD_EMU_FLAGS", "") if flags is None else flags
    if _EMU is None:
        _EMU = {}
    if flags not in _EMU:
        tag = "".join(ch if ch.isalnum() else "_" for ch in flags)
        out_dir = EMU_DIR if os.access(EMU_DIR, os.W_OK) else tempfile.gettempdir()
        so, src = os.path.join(out_dir, f"libbbd_emu{tag}.so"), os.path.join(EMU_DIR, "bbd_emu.cpp")
        csrc = os.path.join(os.path.dirname(EMU_DIR), "..", "baseboostdepth_b200", "csrc")
        deps = [src, os.path.join(EMU_DIR, "simt.h")] + [os.path.join(csrc, f) for f in os.listdir(csrc)]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC"] + flags.split()
                           + ["-o", so, src], check=True)
        _EMU[flags] = _lib.Backend(so, "emu_", cuda=False)
    return _EMU[flags]


def run_fused(inputs, outputs, opt, noise, num_scales, backend=None, groups=None, want_winner=True):
    s_rows = inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None
    plan = plan_for(inputs["ordering"], opt.trimin, opt.decomp, s_rows, groups)
    losses = loss_step(inputs, outputs, opt, plan, noise=noise, num_scales=num_scales, backend=backend,
                       want_winner=want_winner)
    return losses, plan


def to_device(d, device):
    return {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in d.items()}


def mirror_to_device(inputs, outputs, params, device):
    """Copy a CPU batch to the GPU so that the hot path sees *identical* inputs: the camera motions
    are the CPU-assembled matrices (sin/cos differ by ulps between CPU and CUDA, and white-noise
    images amplify an ulp of pose into 1e-4 of warped intensity), fed as leaves.  Returns
    (inputs, outputs, leaves) where leaves maps ("disp", s) / ("cam_T_cam", 0, f) to GPU leaf tensors."""
    gi = to_device(inputs, device)
    go, leaves = {}, {}
    for k, v in outputs.items():
        if k[0] == "disp":
            t = v.detach().to(device).requires_grad_(True)
            go[k], leaves[k] = t, t
        elif k[0] == "cam_T_cam":
            t = v.detach().to(device)
            if t.numel():
                t.requires_grad_(True)
                leaves[k] = t
            go[k] = t
        elif k[0] == "cam_T_cam_error":
            go[k] = v.detach().to(device)
    return gi, go, leaves


def retain_pose_grads(outputs):
    for k, v in outputs.items():
        if k[0] == "cam_T_cam" and v.requires_grad and v.numel():
            v.retain_grad()
