"""Test helpers of the colour-frame gradients: mark, read and check the gradients of a batch's colour tensors."""
from __future__ import annotations

import torch


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
