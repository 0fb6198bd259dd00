"""Fused drop-ins for the reference trainer's loss methods.

``FusedLossMixin`` overrides ``generate_images_pred(inputs, outputs)`` and
``compute_losses(inputs, outputs)`` with the signatures, option handling and
result keys of the reference (``trainer.py:444-475`` and ``:488-570``), so

    class FusedTrainer(FusedLossMixin, trainer.Trainer): pass

trains with the reference's ``process_batch`` / ``run_epoch`` untouched.  The work
itself is ``loss_step`` below: a plan lookup, a tiny batched ``K @ T``, the kernel
launches of ``fused.fused_losses`` (nine forward, five backward) and the loss assembly.

Differences a caller can observe (all deliberate):
  * ``outputs[("depth", 0, s)]`` is filled by ``compute_losses`` (not earlier) and
    carries no autograd graph -- the gradient to the disparity is produced by the
    fused node itself;
  * ``outputs[("color", f, s)]`` / ``("color_D", f, s)`` are only materialised on
    logging steps (``self.early_phase == 0``, ``trainer.py:259-283``) or on request
    (``materialise_warps``), because the loss never needs them in memory;
  * ``self.ident`` (automask statistics, ``trainer.py:547``) holds the same boolean
    planes, derived from the argmin plane the kernel writes, when
    ``self.collect_ident`` is set.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch

from . import _lib, fused
from .fused import _PosePack, combine_losses, fused_losses, pack_poses, start_side_branch
from .plan import LossPlan, build_plan

_PLAN_CACHE: Dict = {}


def plan_for(ordering, trimin: bool, decomp: bool, s_rows: Optional[int] = None, groups=None) -> LossPlan:
    """Cached ``build_plan``: index tables depend only on the batch layout."""
    key = (tuple(tuple(o) for o in ordering), bool(trimin), bool(decomp), s_rows,
           tuple(groups) if groups is not None else None)
    plan = _PLAN_CACHE.get(key)
    if plan is None:
        if len(_PLAN_CACHE) > 4096:
            _PLAN_CACHE.clear()
        plan = build_plan(ordering, trimin=trimin, decomp=decomp, groups=groups, s_stack_rows=s_rows)
        _PLAN_CACHE[key] = plan
    return plan


def _frame_poses(plan: LossPlan, inputs, outputs, key="cam_T_cam", row_masks=None):
    """Per-frame pose stacks aligned with ``plan.sel[f]`` (reference ``trainer.py:463-472``)."""
    T = {}
    for f in plan.frames:
        if f == "s":
            if key != "cam_T_cam":
                continue
            T[f] = inputs["stereo_T"].index_select(0, _index_tensor(plan, ("sel", "s"), plan.sel["s"],
                                                                   inputs["stereo_T"].device))
            continue
        Tf = outputs[(key, 0, f)]
        n = len(plan.sel[f])
        if Tf.shape[0] != n:
            # incremental pose mode keeps one row per sample with baseline >= |f| and masks
            # them with valid_(tri_)mask[|f|] (trainer.py:467-469)
            if row_masks is None or abs(f) not in row_masks or len(row_masks[abs(f)]) != Tf.shape[0]:
                raise ValueError(f"pose stack of frame {f} has {Tf.shape[0]} rows, expected {n}")
            Tf = Tf[row_masks[abs(f)]]
        T[f] = Tf
    return T


def _index_tensor(plan: LossPlan, key, values, device):
    """Small index tensors derived from the plan, uploaded once (keeps steps free of H2D copies so
    that a step can be captured in a CUDA graph)."""
    cache = plan.__dict__.setdefault("_index_cache", {})
    k = (key, str(device))
    t = cache.get(k)
    if t is None:
        t = torch.as_tensor(list(values), device=device, dtype=torch.long)
        cache[k] = t
    return t


def draw_noise(plan: LossPlan, height, width, device, overlap=False):
    """Tie-break noise exactly as the reference draws it: one ``torch.randn`` per group, in
    group order, of the group's plane-stack shape (``trainer.py:518,522``).  Returned raw;
    the ``* 1e-5`` is applied inside the identity kernel (``noise_scale``).

    ``overlap`` (CUDA): the draws run on a helper stream next to the pose packing (same generator, same order,
    hence the same numbers); returns ``(noise, event)`` and the caller makes the launch stream wait for
    ``event`` before the identity pre-pass."""
    shapes = {g: (len(plan.group_members[g]), 1, height, width) for g in plan.groups}
    if not (overlap and torch.device(device).type == "cuda" and fused._USE_SIDE):
        return {g: torch.randn(shapes[g], device=device) for g in plan.groups}, None
    main, side = torch.cuda.current_stream(), fused.noise_stream(torch.device(device))
    noise = {g: torch.empty(shapes[g], device=device) for g in plan.groups}  # allocated on the launch stream
    fork = torch.cuda.Event()
    fork.record(main)
    side.wait_event(fork)
    with torch.cuda.stream(side):
        for g in plan.groups:
            noise[g].normal_()
        done = torch.cuda.Event()
        done.record(side)
    return noise, done


def loss_step(inputs, outputs, opt, plan: Optional[LossPlan] = None, noise=None, num_scales=None,
              backend: Optional[_lib.Backend] = None, want_winner=False, row_masks=None, groups=None,
              timers: Optional[dict] = None):
    """Fused ``generate_images_pred`` + ``compute_losses``: returns the reference's ``losses`` dict.

    ``noise``: per-group planes already scaled by 1e-5 (as the oracle takes them); when
    omitted they are drawn like the reference does.  Also stores ``("depth",0,s)`` in
    ``outputs`` and, with ``want_winner``, ``outputs["argmin"]`` (S,B,H,W) uint8.
    """
    ordering = inputs["ordering"]
    color0 = inputs[("color", 0, 0)]
    B, _, H, W = color0.shape
    if plan is None:
        s_rows = inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None
        plan = plan_for(ordering, opt.trimin, opt.decomp, s_rows, groups)
    scales = list(opt.scales)
    num_scales = num_scales if num_scales is not None else len(scales)

    disps = [outputs[("disp", s)] for s in scales]
    pyramid = [inputs[("color", 0, s)] for s in scales]
    if getattr(opt, "SQL", False):
        for d, c in zip(disps, pyramid):
            if d.shape[-2:] != c.shape[-2:]:
                raise NotImplementedError("opt.SQL with a disparity pyramid smaller than its colour level")
    # disparity -> depth and the smoothness kernels start first, on the helper stream; the pose packing,
    # the noise draw and the identity pre-pass below run next to them
    be = backend if backend is not None else _lib.cuda_backend()
    noise_ready = None
    if noise is None:
        noise, noise_ready = draw_noise(plan, H, W, color0.device, overlap=be.cuda)
        noise_scale = 0.00001
    else:
        noise_scale = 1.0
    # (a colour level that requires grad also needs the smoothness normalisation scalars)
    pre = start_side_branch(be, disps, pyramid, (B, H, W), opt.min_depth, opt.max_depth, getattr(opt, "SQL", False),
                            torch.is_grad_enabled(), timers=timers,
                            need_coef=torch.is_grad_enabled() and any(p.requires_grad for p in pyramid))

    T = _frame_poses(plan, inputs, outputs, "cam_T_cam", row_masks)
    T_err = _frame_poses(plan, inputs, outputs, "cam_T_cam_error", row_masks) if plan.decomp else None
    P = pack_poses(plan, inputs[("K", 0)], T, T_err, backend=backend)
    frames = {f: inputs[("color", f, 0)] for f in plan.frames}
    if noise_ready is not None:
        torch.cuda.current_stream().wait_event(noise_ready)

    reproj, smooth, aux = fused_losses(
        plan, color0, frames, disps, inputs[("inv_K", 0)], P, noise, pyramid,
        min_depth=opt.min_depth, max_depth=opt.max_depth, no_ssim=opt.no_ssim,
        sql=getattr(opt, "SQL", False), noise_scale=noise_scale, want_winner=want_winner, backend=backend,
        timers=timers, pre=pre)

    weights = _weights(tuple(opt.disparity_smoothness / (2 ** s) for s in scales), reproj.device)
    per_scale, total = combine_losses(reproj, smooth, weights, num_scales, backend=backend)
    losses = {f"loss/{s}": per_scale[i] for i, s in enumerate(scales)}
    losses["loss"] = total
    for i, s in enumerate(scales):
        outputs[("depth", 0, s)] = aux["depth"][i].unsqueeze(1)
    if want_winner:
        outputs["argmin"] = aux["winner"]
    return losses


_WEIGHT_CACHE: Dict = {}


def _weights(values, device):
    key = (values, str(device))
    w = _WEIGHT_CACHE.get(key)
    if w is None:
        w = torch.tensor(values, dtype=torch.float32, device=device)
        _WEIGHT_CACHE[key] = w
    return w


def materialise_warps(inputs, outputs, opt, plan: LossPlan, scales=None, backend: Optional[_lib.Backend] = None,
                      row_masks=None):
    """Fill ``outputs[("color", f, s)]`` (and ``("color_D", f, s)``) like ``trainer.py:434-442``.

    One launch per (frame, scale); used on logging steps and by the parity tests.
    """
    be = backend if backend is not None else _lib.cuda_backend()
    color0 = inputs[("color", 0, 0)]
    B, _, H, W = color0.shape
    scales = list(opt.scales) if scales is None else scales
    K, inv_K = inputs[("K", 0)], inputs[("inv_K", 0)].contiguous()
    T = _frame_poses(plan, inputs, outputs, "cam_T_cam", row_masks)
    T_err = _frame_poses(plan, inputs, outputs, "cam_T_cam_error", row_masks) if plan.decomp else {}
    for s in scales:
        depth = outputs[("depth", 0, s)].detach()
        for f in plan.frames:
            n = len(plan.sel[f])
            rows = _index_tensor(plan, ("rows", f), plan.stack_row[f], color0.device)
            sel = _index_tensor(plan, ("sel", f), plan.sel[f], color0.device)
            images = inputs[("color", f, 0)].index_select(0, rows).contiguous()
            d = depth.index_select(0, sel).contiguous()
            for key, poses in (("color", T), ("color_D", T_err)):
                if f not in poses:
                    continue
                if n:
                    k_row = torch.arange(n, dtype=torch.int32, device=color0.device)
                    P = _PosePack.apply(poses[f].detach(), K, k_row, be)
                else:
                    P = K.new_zeros(0, 3, 4)
                warped = torch.empty_like(images)
                be.check_device(images, d, P)
                if n:
                    be.call("warp_forward", n, H, W, C.c_void_p(images.data_ptr()), C.c_void_p(d.data_ptr()),
                            C.c_void_p(inv_K.data_ptr()), C.c_void_p(P.data_ptr()), C.c_void_p(warped.data_ptr()),
                            C.c_void_p(None))
                outputs[(key, f, s)] = warped
    return outputs


class FusedLossMixin:
    """Mix into the reference ``Trainer`` (left of it in the MRO) to use the fused path."""

    collect_ident = False     # fill self.ident like trainer.py:547 (costs an argmin plane write)
    always_warp = False       # materialise ("color", f, s) every step, not only when logging
    _bbd_backend = None       # tests point this at the CPU harness; None = the CUDA library

    def _bbd_plan(self, inputs) -> LossPlan:
        s_rows = inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None
        return plan_for(inputs["ordering"], self.opt.trimin, self.opt.decomp, s_rows)

    def _bbd_row_masks(self):
        return self.valid_tri_mask if self.opt.trimin else self.valid_mask

    def generate_images_pred(self, inputs, outputs):
        """Reference ``trainer.py:444-475``.  The warps are folded into ``compute_losses``;
        here only the batch plan is prepared (and remembered for the logging hook)."""
        self._bbd_current_plan = self._bbd_plan(inputs)
        return outputs

    def compute_losses(self, inputs, outputs):
        """Reference ``trainer.py:488-570``: returns ``{"loss", "loss/<s>"...}``."""
        plan = getattr(self, "_bbd_current_plan", None) or self._bbd_plan(inputs)
        want = bool(self.collect_ident and self.opt.trimin)
        losses = loss_step(inputs, outputs, self.opt, plan, num_scales=self.num_scales, want_winner=want,
                           row_masks=self._bbd_row_masks(), backend=self._bbd_backend)
        if want:
            self.ident = ident_statistics(plan, outputs["argmin"][-1])
        if self.always_warp or getattr(self, "early_phase", 1) == 0:
            with torch.no_grad():
                materialise_warps(inputs, outputs, self.opt, plan, row_masks=self._bbd_row_masks(),
                                  backend=self._bbd_backend)
        return losses


def ident_statistics(plan: LossPlan, winner: torch.Tensor):
    """``(dictor_norm, dictor_guide)`` of ``Trainer.x_min_opt`` (``trainer.py:983-1100``) from the
    argmin plane of the last scale: per group, where a warped (resp. error-induced) candidate won."""
    norm = {(g, "norm"): [] for g in plan.baselines}
    guide = {(g, "guide"): [] for g in plan.baselines}
    for g in plan.groups:
        members = plan.group_members[g]
        if not members:
            continue
        idx = torch.as_tensor(members, device=winner.device, dtype=torch.long)
        w = winner.index_select(0, idx)
        n_src = len([1 for f, err in plan.rep[members[0]] if not err])
        n_rep = len(plan.rep[members[0]])
        norm[(g, "norm")].append(w < n_src)
        if plan.decomp and g != "s":
            guide[(g, "guide")].append((w >= n_src) & (w < n_rep))
    return norm, guide
