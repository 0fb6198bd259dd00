"""Test plumbing of the colour-frame gradients: the CPU harness with the frame-gradient entry points, and
helpers that mark, read and check the gradients of a batch's colour tensors."""
from __future__ import annotations

import os
import subprocess
import tempfile

import torch

from baseboostdepth_b200 import _lib
from fused_util import EMU_DIR

_EMU = None


def emu_frame_backend() -> _lib.Backend:
    """Compile (if stale) and load the CPU harness of tests/emu/bbd_emu.cpp together with the emu_* versions of
    the frame-gradient entry points (tests/emu/bbd_emu_framegrad.cpp).  Built next to the sources, or in the
    temporary directory when the tree is read-only."""
    global _EMU
    if _EMU is None:
        src = os.path.join(EMU_DIR, "bbd_emu_framegrad.cpp")
        out_dir = EMU_DIR if os.access(EMU_DIR, os.W_OK) else tempfile.gettempdir()
        so = os.path.join(out_dir, "libbbd_emu_framegrad.so")
        csrc = os.path.join(os.path.dirname(EMU_DIR), "..", "baseboostdepth_b200", "csrc")
        deps = [src, os.path.join(EMU_DIR, "bbd_emu.cpp"), os.path.join(EMU_DIR, "simt.h")] + [
            os.path.join(csrc, f) for f in os.listdir(csrc)]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-mfma", "-shared", "-fPIC", "-o", so, src],
                           check=True)
        _EMU = _lib.Backend(so, "emu_", cuda=False)
    return _EMU


def frame_keys(inputs):
    """Every colour tensor of a batch: the target, the source stacks ("color", f, 0) and the pyramid levels."""
    return sorted((k for k in inputs if isinstance(k, tuple) and k[0] == "color"), key=str)


def require_frame_grads(inputs, keys=None):
    """Set requires_grad on the colour tensors named by `keys` (default: all of them)."""
    for k in (frame_keys(inputs) if keys is None else keys):
        inputs[k].requires_grad_(True)


def frame_grad(inputs, k):
    """.grad of a colour tensor, zeros where autograd left None (a stack the loss never reads)."""
    t = inputs[k]
    return t.grad if t.grad is not None else torch.zeros_like(t)


def referenced_rows(plan):
    """{frame: set of stack rows} that some warped or identity candidate of the plan reads."""
    used = {f: set() for f in plan.frames}
    for b in range(plan.batch):
        n_rep, n_id = int(plan.hdr[b, 0]), int(plan.hdr[b, 1])
        for k in range(n_rep):
            used[plan.frames[int(plan.rep_tab[b, k, 0])]].add(int(plan.rep_tab[b, k, 1]))
        for j in range(n_id):
            used[plan.frames[int(plan.ident_tab[b, j, 0])]].add(int(plan.ident_tab[b, j, 1]))
    return used
