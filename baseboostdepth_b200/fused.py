"""Fused view-synthesis loss: one autograd node over the C ABI.

``fused_losses`` evaluates, for all scales of a step, what the reference spreads
over ``generate_images_pred`` (``trainer.py:444-475``) and ``compute_losses``
(``trainer.py:488-570``): disparity -> depth, identity pre-pass, warp + SSIM/L1 +
per-pixel minimum, smoothness -- forward *and* backward -- in a dozen kernel
launches (the small ones on helper streams next to the identity pre-pass), and returns the per-scale reprojection means and smoothness terms as
differentiable tensors.  Gradients flow to the disparities and to the packed
projection matrices ``P = (K @ T)[:, :3, :]``, and to the colour frames (target,
source stacks, pyramid levels) that require one (``_frame_backward``).

Because every loss term is a mean with a weight known in advance, the kernels
produce the unit gradients during the forward launch; ``backward`` only folds
the upstream scalars in while gathering the full-resolution depth gradient
down to the disparity resolution.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib
from .plan import LossPlan


import os as _os

# BBD_SIDE_STREAMS=0 keeps every kernel on the launch stream (debugging / A-B measurements)
_USE_SIDE = _os.environ.get("BBD_SIDE_STREAMS", "1") != "0"
# 1: the two-pass transpose of the upsample, its full-resolution level on a helper stream (round 1); default: the
# single-launch form (bbd_disp_to_depth_backward picks it whenever every level is a 1/2/4/8 reduction)
_SPLIT_D2D_BACKWARD = _os.environ.get("BBD_D2D_SPLIT", "0") != "0"
# BBD_FORCE_TILE=1 pins the round-1 tile kernel (every elementary operation rounded like the reference's
# separate ATen kernels) instead of the streaming kernel with contracted / separable arithmetic
_FORCE_TILE = _os.environ.get("BBD_FORCE_TILE", "0") != "0"
_SIDE: Dict = {}


def _side_streams(device):
    """Two helper streams per device: the disparity -> depth kernel on one, the smoothness kernels on the
    other (all small and latency-bound) run next to the identity pre-pass and join the launch stream
    before the fused kernel."""
    s = _SIDE.get(device)
    if s is None:
        s = _SIDE[device] = (torch.cuda.Stream(device=device), torch.cuda.Stream(device=device))
    return s


def _pose_rows_covered(plan) -> bool:
    c = getattr(plan, "_pose_rows_covered", None)
    if c is None:
        used = set()
        for b in range(plan.batch):
            for k in range(int(plan.hdr[b, 0])):
                used.add(int(plan.rep_tab[b, k, 2]))
        c = used == set(range(plan.n_pose))
        try:
            object.__setattr__(plan, "_pose_rows_covered", c)
        except Exception:
            pass
    return c


_NOISE_STREAM: Dict = {}


def noise_stream(device):
    """Helper stream of the tie-break noise draws (trainer.draw_noise)."""
    s = _NOISE_STREAM.get(device)
    if s is None:
        s = _NOISE_STREAM[device] = torch.cuda.Stream(device=device)
    return s


def _call(be, timers, key, name, *args):
    """``be.call`` with an optional pair of CUDA events around it on the stream it is enqueued on
    (bench.py's per-kernel table); ``timers[key]`` = (start, end)."""
    if timers is None or not be.cuda:
        be.call(name, *args)
        return
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    be.call(name, *args)
    t1.record()
    timers[key] = (t0, t1)


_TICKETS: Dict = {}


def _tickets(device, n):
    """Zero-initialised int32 counters of the fused finalize; the kernel leaves them zero after every launch."""
    key = (str(device), n)
    t = _TICKETS.get(key)
    if t is None:
        t = _TICKETS[key] = torch.zeros(n, device=device, dtype=torch.int32)
    return t


def _tables(plan: LossPlan, device):
    cache = getattr(plan, "_dev_tables", None)
    if cache is None or cache[0] != str(device):
        hdr = torch.from_numpy(plan.hdr).to(device)
        rep = torch.from_numpy(plan.rep_tab).to(device)
        ident = torch.from_numpy(plan.ident_tab).to(device)
        cache = (str(device), hdr, rep, ident)
        plan._dev_tables = cache
    t = _lib.Tables()
    t.hdr, t.rep, t.ident = cache[1].data_ptr(), cache[2].data_ptr(), cache[3].data_ptr()
    return t


def _frame_ptrs(plan: LossPlan, frames: Dict, height, width):
    arr = (C.c_void_p * _lib.MAX_FRAMES)()
    keep = []
    for slot, f in enumerate(plan.frames):
        t = frames[f]
        need = max(plan.stack_row[f], default=-1) + 1
        if t.shape[0] < need or tuple(t.shape[1:]) != (3, height, width):
            raise ValueError(f"frame stack {f!r} has shape {tuple(t.shape)}, need >= {need} rows of (3,{height},{width})")
        t = t.contiguous()
        keep.append(t)
        arr[slot] = t.data_ptr() if t.numel() else None
    return arr, keep


def stream_eligible(plan: LossPlan) -> bool:
    """The streaming kernel serves every batch layout (one or two candidates per sample in one sweep, more in
    sweeps over candidate pairs); BBD_FORCE_TILE=1 pins the tile kernel."""
    n = [len(r) for r in plan.rep]
    return (not _FORCE_TILE) and min(n) >= 1 and max(n) <= _lib.MAX_REP


def rgba_buffers(keep, height, width):
    """Channel-interleaved copies of the frame stacks: one 16-byte load then fetches a bilinear tap of all
    three channels.  Only allocated here; the identity pre-pass fills them while it reads the frames."""
    arr = (C.c_void_p * _lib.MAX_FRAMES)()
    owned = []
    for slot, t in enumerate(keep):
        if not t.numel():
            continue
        out = torch.empty(t.shape[0], height, width, 4, device=t.device, dtype=torch.float32)
        owned.append(out)
        arr[slot] = out.data_ptr()
    return arr, owned


def disps_key(disps):
    """Identity of a disparity list (a started side branch is valid for exactly this memory)."""
    return tuple((d.data_ptr(), tuple(d.shape), d._version) for d in disps)


def start_side_branch(be, disps, pyramid, bhw, min_depth, max_depth, sql, need_grad, timers=None, need_coef=False):
    """Launch disparity -> depth (reference ``trainer.py:456`` + ``layers.py:13-22``) and the smoothness
    kernels (``trainer.py:560-564``) for one step.  They depend only on the disparities and the colour
    pyramid, are small and latency-bound, and therefore run on a helper stream between a fork and a
    join event (graph-capturable) while the launch stream goes on with the pose packing, the noise
    draw and the identity pre-pass; ``_FusedLoss.forward`` waits for ``join`` before the fused kernel.
    Every buffer is allocated here on the launch stream, before the fork.  ``need_coef``: keep the
    per-(level, sample) normalisation scalars even without disparity gradients (the pyramid's gradient
    reads them)."""
    B, H, W = bhw
    S = len(disps)
    assert 1 <= S <= _lib.MAX_SCALES
    be.check_device(*disps, *pyramid)
    if need_grad:
        # the transpose of the upsample is implemented for the pyramid the networks produce (integer factors
        # up to 8); say so here rather than from inside autograd.backward
        for d in disps:
            h, w = d.shape[-2:]
            if H % h or W % w or H // h > 8 or W // w > 8:
                raise NotImplementedError(f"bbd: disparity level {tuple(d.shape[-2:])} is not an integer factor <= 8 "
                                          f"of the frame {(H, W)}; gradients are only provided for such pyramids")
    dev = disps[0].device
    f32 = dict(device=dev, dtype=torch.float32)
    disps_c = [d.detach().contiguous() for d in disps]
    keep = []
    depth = torch.empty(S, B, H, W, **f32)
    d2d = _lib.D2DArgs()
    d2d.batch, d2d.levels, d2d.height, d2d.width = B, S, H, W
    d2d.min_disp = 1 / max_depth
    d2d.disp_span = 1 / min_depth - 1 / max_depth
    d2d.sql = int(sql)
    for l, d in enumerate(disps_c):
        d2d.h[l], d2d.w[l] = d.shape[2], d.shape[3]
        d2d.disp[l] = d.data_ptr()
    d2d.depth = depth.data_ptr()

    sa = _lib.SmoothArgs()
    sa.batch, sa.levels, sa.normalize = B, S, 1
    gsm = []
    for l, d in enumerate(disps_c):
        img = pyramid[l].contiguous()
        keep.append(img)
        assert img.shape[0] == B and img.shape[-2:] == d.shape[-2:], (img.shape, d.shape)
        sa.h[l], sa.w[l] = d.shape[2], d.shape[3]
        sa.disp[l], sa.img[l] = d.data_ptr(), img.data_ptr()
        if need_grad:
            g = torch.empty_like(d)
            gsm.append(g)
            sa.gdisp[l] = g.data_ptr()
    hs = (C.c_int32 * S)(*[d.shape[2] for d in disps_c])
    ws = (C.c_int32 * S)(*[d.shape[3] for d in disps_c])
    scratch = torch.empty(max(1, be.value("smooth_scratch_floats", B, S, hs, ws)), **f32)
    smooth = torch.empty(S, **f32)
    sa.scratch, sa.loss = scratch.data_ptr(), smooth.data_ptr()
    keep.append(scratch)
    # the mean-normalisation of the smoothness gradient is finished by the disparity backward (one pass less)
    coef = torch.empty(S, B, 2, **f32) if need_grad or need_coef else None
    if coef is not None:
        sa.defer_norm, sa.coef = 1, coef.data_ptr()

    join = None
    if be.cuda and _USE_SIDE:
        main, (side_a, side_b) = torch.cuda.current_stream(), _side_streams(dev)
        fork = torch.cuda.Event()
        fork.record(main)
        join = []
        for side, name, args in ((side_a, "smooth_fused", sa), (side_b, "disp_to_depth_forward", d2d)):
            side.wait_event(fork)
            with torch.cuda.stream(side):
                _call(be, timers, name, name, C.byref(args))
                ev = torch.cuda.Event()
                ev.record(side)
                join.append(ev)
        # (joining the smoothness kernels only after the fused kernel was measured: their tail then
        # competes with its first waves and costs it 9 us -- no net gain)
    else:
        _call(be, timers, "disp_to_depth_forward", "disp_to_depth_forward", C.byref(d2d))
        _call(be, timers, "smooth_fused", "smooth_fused", C.byref(sa))
    return dict(disps=disps_key(disps), disps_c=disps_c, d2d=d2d, depth=depth, gsm=gsm, smooth=smooth, join=join,
                keep=keep, coef=coef)


class _FusedLoss(torch.autograd.Function):
    """(P, disp_0..disp_{S-1}, target, frame stacks in plan.frames order, pyramid_0..pyramid_{S-1})
    -> (reproj[S], smooth[S]); inv_K and the noise are closed over."""

    @staticmethod
    def forward(ctx, cfg, P, *tensors):
        be: _lib.Backend = cfg["backend"]
        plan: LossPlan = cfg["plan"]
        target, frames, inv_K = cfg["target"], cfg["frames"], cfg["inv_K"]
        noise, pyramid = cfg["noise"], cfg["pyramid"]
        disps = tensors[:len(pyramid)]
        B, _, H, W = target.shape
        S = len(disps)
        dev = target.device
        need_grad = bool(cfg["need_grad"])
        frame_grad = bool(cfg["frame_grad"])
        f32 = dict(device=dev, dtype=torch.float32)
        be.check_device(target, inv_K, P, *disps, *pyramid, *noise.values(), *frames.values())
        assert plan.batch == B and P.shape == (plan.n_pose, 3, 4), (P.shape, plan.n_pose)
        assert S <= _lib.MAX_SCALES

        Pc = P.detach().contiguous()
        target = target.contiguous()
        inv_K = inv_K.contiguous()
        tab = _tables(plan, dev)
        frame_arr, keep = _frame_ptrs(plan, frames, H, W)
        frames_c = list(keep)
        rgba_arr, rgba_keep = rgba_buffers(keep, H, W) if stream_eligible(plan) else (None, [])

        # 1 + 5. disparity -> depth and smoothness: on the helper stream (started here unless the caller
        # already did, see start_side_branch)
        # (popped: `smooth` becomes an output of this node, and an output reachable from ctx would be a
        # reference cycle that keeps the autograd graph -- and its AccumulateGrad nodes -- alive)
        pre = cfg.pop("pre", None)
        pyr_grad = frame_grad and any(p.requires_grad for p in pyramid)
        if (pre is None or pre["disps"] != disps_key(disps) or (need_grad and not pre["gsm"])
                or (pyr_grad and pre["coef"] is None)):
            pre = start_side_branch(be, disps, pyramid, (B, H, W), cfg["min_depth"], cfg["max_depth"], cfg["sql"],
                                    need_grad, timers=cfg.get("timers"), need_coef=pyr_grad)
        disps_c, d2d, depth, gsm, smooth, join = (pre[k] for k in ("disps_c", "d2d", "depth", "gsm", "smooth", "join"))
        keep.extend(pre["keep"])

        # 2. identity pre-pass (once per step)
        ident_min = torch.empty(B, H, W, **f32)
        want_winner = bool(cfg["want_winner"]) or frame_grad   # the frame gradient differentiates these winners
        ident_arg = torch.empty(B, H, W, device=dev, dtype=torch.uint8) if want_winner else None
        ia = _lib.IdentArgs()
        ia.batch, ia.height, ia.width, ia.no_ssim = B, H, W, int(cfg["no_ssim"])
        ia.target = target.data_ptr()
        ia.frames = frame_arr
        for slot, g in enumerate(plan.groups):
            n = noise[g].contiguous()
            keep.append(n)
            assert n.shape[0] == len(plan.group_members[g]) and tuple(n.shape[-2:]) == (H, W)
            ia.noise[slot] = n.data_ptr()
        ia.noise_scale = float(cfg["noise_scale"])
        ia.tab = tab
        ia.ident_min = ident_min.data_ptr()
        ia.ident_arg = _lib.ptr(ident_arg)
        if rgba_arr is not None:
            ia.frames_rgba = rgba_arr
        ia.force_tile = int(_FORCE_TILE)
        _call(be, cfg.get("timers"), "ident_forward", "ident_forward", C.byref(ia))
        for ev in join or ():
            torch.cuda.current_stream().wait_event(ev)

        # 3. fused warp + photometric + min (+ gradients)
        ntiles = be.value("reproj_tiles", H, W)
        loss_part = torch.empty(S, B, ntiles, **f32)
        gpose_part = torch.empty(S, B, _lib.MAX_REP, ntiles, 12, **f32) if need_grad else None
        gdepth = torch.empty(S, B, H, W, **f32) if need_grad else None
        # batches with more than two candidates per sample run as a selection launch and a gradient launch that reads the
        # per-pixel winners: the plane is needed even when the caller does not ask for it
        need_winner = want_winner or (need_grad and plan.max_rep > 2 and rgba_arr is not None)
        winner = torch.empty(S, B, H, W, device=dev, dtype=torch.uint8) if need_winner else None
        ra = _lib.ReprojArgs()
        ra.batch, ra.height, ra.width, ra.num_scales = B, H, W, S
        ra.no_ssim, ra.need_grad, ra.max_rep, ra.num_pose = int(cfg["no_ssim"]), int(need_grad), plan.max_rep, plan.n_pose
        ra.target, ra.frames, ra.depth = target.data_ptr(), frame_arr, depth.data_ptr()
        ra.inv_K, ra.P, ra.ident_min, ra.tab = inv_K.data_ptr(), Pc.data_ptr(), ident_min.data_ptr(), tab
        ra.loss_part, ra.gpose_part, ra.gdepth = loss_part.data_ptr(), _lib.ptr(gpose_part), _lib.ptr(gdepth)
        ra.winner, ra.ident_arg = _lib.ptr(winner), _lib.ptr(ident_arg)
        if rgba_arr is not None:
            ra.frames_rgba = rgba_arr
        ra.min_rep, ra.force_tile = min(len(r) for r in plan.rep), int(_FORCE_TILE)
        # the streaming kernel reduces its own partials (last warp of every (scale, sample), fixed order)
        reproj = torch.empty(S, **f32)
        # every pose row belongs to exactly one (sample, candidate) of the tables, so the reduction writes all of
        # gpose: no zero fill on the critical path (checked once per plan; a plan with orphan rows gets zeros)
        gpose = None
        if need_grad:
            gpose = (torch.empty if _pose_rows_covered(plan) else torch.zeros)(S, plan.n_pose, 3, 4, **f32)
        fused_finalize = rgba_arr is not None and plan.max_rep <= 2
        if fused_finalize:
            ra.tickets = _tickets(dev, S * B + S).data_ptr()
            pair_sum = torch.empty(S * B, **f32)
            ra.pair_sum, ra.loss_out, ra.gpose_out = pair_sum.data_ptr(), reproj.data_ptr(), _lib.ptr(gpose)
        timers = cfg.get("timers")
        _call(be, timers, "reproj_fused", "reproj_fused", C.byref(ra))
        if timers is not None and be.cuda:
            timers["reproj_kernel_name"] = be.dll.bbd_reproj_kernel_name(C.byref(ra)).decode()

        # 4. fixed-order reduction of the per-tile partials (tile kernel; the streaming kernel has done it)
        if not (fused_finalize and be.value("reproj_finalizes_itself", C.byref(ra))):
            _call(be, timers, "reproj_finalize", "reproj_finalize", C.byref(ra), C.c_void_p(reproj.data_ptr()),
                  C.c_void_p(_lib.ptr(gpose)))

        ctx.cfg = cfg
        ctx.d2d = d2d
        del rgba_keep   # consumed by the fused kernel (stream-ordered: the allocator may reuse it from here on)
        ctx.keep = (disps_c, depth, gdepth, gpose, gsm, pre["coef"])
        ctx.aux = {"depth": depth, "ident_min": ident_min, "ident_arg": ident_arg, "winner": winner}
        ctx.frame_grad = frame_grad
        if frame_grad:
            # what the frame gradient reads again: the argument block of the fused kernel and the buffers it points at
            ctx.frame_keep = (ra, target, inv_K, Pc, frames_c, pre["keep"][:S], winner, ident_arg, ident_min)
        cfg["aux"] = ctx.aux
        return reproj, smooth

    @staticmethod
    def backward(ctx, g_reproj, g_smooth):
        cfg = ctx.cfg
        be: _lib.Backend = cfg["backend"]
        disps_c, depth, gdepth, gpose, gsm, coef = ctx.keep
        g_reproj = g_reproj.contiguous().float()
        g_smooth = g_smooth.contiguous().float()
        S = len(disps_c)
        frame_grads = _frame_backward(ctx, be, g_reproj, g_smooth, S) if ctx.frame_grad else (None,) * (
            len(ctx.needs_input_grad) - 2 - S)
        if gdepth is None:
            if not ctx.frame_grad:
                raise RuntimeError("bbd: fused loss was evaluated with need_grad=False")
            return (None, None) + (None,) * S + frame_grads
        gP = torch.einsum("s,spij->pij", g_reproj, gpose) if ctx.needs_input_grad[1] else None
        d2d = ctx.d2d
        gdisps = [torch.empty_like(d) for d in disps_c]
        d2d.gdepth = gdepth.data_ptr()
        d2d.gscale = g_reproj.data_ptr()
        d2d.gsmooth_scale = g_smooth.data_ptr()
        d2d.gsmooth_coef = _lib.ptr(coef)
        for l, g in enumerate(gdisps):
            d2d.gdisp[l] = g.data_ptr()
            d2d.gsmooth[l] = gsm[l].data_ptr()
        scratch = torch.empty(max(1, be.value("d2d_scratch_floats", C.byref(d2d))), device=gdepth.device,
                              dtype=torch.float32)
        d2d.scratch = scratch.data_ptr()
        full_res_first = S > 1 and tuple(disps_c[0].shape[-2:]) == tuple(depth.shape[-2:])
        timers = cfg.get("timers")
        if timers is not None and be.cuda:
            tb0, tb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tb0.record()
        if be.cuda and full_res_first and _USE_SIDE and _SPLIT_D2D_BACKWARD:
            # pass 2 of a full-resolution level does not read the row sums of pass 1: it runs on a helper
            # stream next to pass 1, the remaining levels follow pass 1 on this stream
            main, (side, _) = torch.cuda.current_stream(), _side_streams(gdepth.device)
            fork = torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)
            with torch.cuda.stream(side):
                be.call("disp_to_depth_backward_pass2", C.byref(d2d), 0, 1)
                join = torch.cuda.Event()
                join.record(side)
            be.call("disp_to_depth_backward_pass1", C.byref(d2d))
            be.call("disp_to_depth_backward_pass2", C.byref(d2d), 1, S)
            main.wait_event(join)
        else:
            be.call("disp_to_depth_backward", C.byref(d2d))
        if timers is not None and be.cuda:
            tb1.record()
            timers["disp_to_depth_backward"] = (tb0, tb1)
        return (None, gP) + tuple(gdisps) + frame_grads


def _frame_backward(ctx, be, g_reproj, g_smooth, S):
    """Gradients of (target, frame stacks..., pyramid levels...) as ``ctx.needs_input_grad`` asks for them:
    bbd_frame_grad, a stable sort of its keys, bbd_frame_grad_stacks, and bbd_smooth_image_grad."""
    cfg = ctx.cfg
    plan: LossPlan = cfg["plan"]
    ra, target, inv_K, Pc, frames_c, pyr_c, winner, ident_arg, ident_min = ctx.frame_keep
    needs = ctx.needs_input_grad[2 + S:]
    n_f = len(frames_c)
    need_target, need_frames, need_pyr = needs[0], needs[1:1 + n_f], needs[1 + n_f:]
    B, _, H, W = target.shape
    dev, HW = target.device, H * W
    f32 = dict(device=dev, dtype=torch.float32)
    gtarget, gframes, gpyr = None, [None] * n_f, [None] * S
    if need_target or any(need_frames):
        fa = _lib.FrameGradArgs()
        fa.gscale = g_reproj.data_ptr()
        for slot, t in enumerate(frames_c):
            fa.stack_rows[slot] = t.shape[0]
        coef = None if cfg["no_ssim"] else torch.empty(S, B, 3, 6, H, W, **f32)
        gpred = torch.empty(S, B, plan.max_rep, 3, H, W, **f32)
        keys = torch.empty(S * B * plan.max_rep * HW, device=dev, dtype=torch.int32)
        gident = torch.empty(B, _lib.MAX_IDENT, 3, H, W, **f32)
        gtarget = torch.empty(B, 3, H, W, **f32) if need_target else None
        fa.coef, fa.gpred, fa.keys = _lib.ptr(coef), gpred.data_ptr(), keys.data_ptr()
        fa.gident, fa.gtarget = gident.data_ptr(), _lib.ptr(gtarget)
        be.call("frame_grad", C.byref(ra), C.byref(fa))
        if any(need_frames):
            keys_sorted, order = torch.sort(keys, stable=True)
            order = order.to(torch.int32)
            seg = torch.empty(sum(t.shape[0] for t in frames_c) * HW + 1, device=dev, dtype=torch.int32)
            fa.keys_sorted, fa.order, fa.seg_start = keys_sorted.data_ptr(), order.data_ptr(), seg.data_ptr()
            for slot, t in enumerate(frames_c):
                if need_frames[slot]:
                    gframes[slot] = torch.empty_like(t) if t.numel() else torch.zeros_like(t)
                    fa.gframes[slot] = _lib.ptr(gframes[slot]) if t.numel() else None
            be.call("frame_grad_stacks", C.byref(ra), C.byref(fa))
    if any(need_pyr):
        _, _, _, _, _, coef_s = ctx.keep
        disps_c = ctx.keep[0]
        sa = _lib.SmoothImgArgs()
        sa.batch, sa.levels = B, S
        sa.coef, sa.gscale = coef_s.data_ptr(), g_smooth.data_ptr()
        for l in range(S):
            sa.h[l], sa.w[l] = disps_c[l].shape[2], disps_c[l].shape[3]
            sa.disp[l], sa.img[l] = disps_c[l].data_ptr(), pyr_c[l].data_ptr()
            if need_pyr[l]:
                gpyr[l] = torch.empty_like(pyr_c[l])
                sa.gimg[l] = gpyr[l].data_ptr()
        be.call("smooth_image_grad", C.byref(sa))
    return (gtarget,) + tuple(gframes) + tuple(gpyr)


def fused_losses(plan: LossPlan, target: torch.Tensor, frames: Dict, disps: Sequence[torch.Tensor],
                 inv_K: torch.Tensor, P: torch.Tensor, noise: Dict, pyramid: Sequence[torch.Tensor], *,
                 min_depth=0.1, max_depth=100.0, no_ssim=False, sql=False, noise_scale=1.0,
                 want_winner=False, need_grad: Optional[bool] = None, backend: Optional[_lib.Backend] = None,
                 timers: Optional[dict] = None, pre: Optional[dict] = None):
    """Per-scale ``(reproj[S], smooth[S], aux)`` of the view-synthesis loss.

    ``frames[f]`` are the compacted ``("color", f, 0)`` stacks, ``disps[s]`` the network
    disparities, ``P`` the packed ``(K @ T)[:, :3, :]`` rows in ``plan.pose_slices()`` order,
    ``noise[g]`` the per-group tie-break planes (multiplied by ``noise_scale`` in-kernel),
    ``pyramid[s]`` the target colour pyramid ``("color", 0, s)``.
    ``aux`` exposes ``depth`` (S,B,H,W) and, with ``want_winner``, the argmin planes.
    """
    be = backend if backend is not None else _lib.cuda_backend()
    if need_grad is None:
        need_grad = torch.is_grad_enabled() and (P.requires_grad or any(d.requires_grad for d in disps))
    frame_list = [frames[f] for f in plan.frames]
    pyramid = list(pyramid)
    frame_grad = torch.is_grad_enabled() and any(t.requires_grad for t in [target] + frame_list + pyramid)
    cfg = dict(backend=be, plan=plan, target=target, frames=frames, inv_K=inv_K, noise=noise,
               pyramid=pyramid, min_depth=min_depth, max_depth=max_depth, no_ssim=no_ssim, sql=sql,
               noise_scale=noise_scale, want_winner=want_winner, need_grad=need_grad, frame_grad=frame_grad,
               timers=timers, pre=pre)
    reproj, smooth = _FusedLoss.apply(cfg, P, *disps, target, *frame_list, *pyramid)
    return reproj, smooth, cfg["aux"]


class _Combine(torch.autograd.Function):
    """(reproj[S], smooth[S]) -> (per_scale[S], total): the loss assembly of ``trainer.py:557-570`` as one
    launch each way instead of ~10 four-element tensor kernels."""

    @staticmethod
    def forward(ctx, reproj, smooth, weight, num_scales, be):
        S = reproj.shape[0]
        r, m = reproj.detach().contiguous(), smooth.detach().contiguous()
        be.check_device(r, m, weight)
        out = torch.empty(S + 1, device=r.device, dtype=torch.float32)   # [per_scale..., total]
        per_scale, total = out[:S], out[S]
        be.call("loss_combine_forward", S, C.c_void_p(r.data_ptr()), C.c_void_p(m.data_ptr()),
                C.c_void_p(weight.data_ptr()), C.c_float(float(num_scales)), C.c_void_p(out.data_ptr()),
                C.c_void_p(out.data_ptr() + 4 * S))
        ctx.weight, ctx.num_scales, ctx.be, ctx.S = weight, float(num_scales), be, S
        ctx.set_materialize_grads(False)    # an unused output arrives as None, not as a zero tensor
        return per_scale, total

    @staticmethod
    def backward(ctx, g_per_scale, g_total):
        S, be = ctx.S, ctx.be
        if g_per_scale is None and g_total is None:
            return None, None, None, None, None
        gps = g_per_scale.contiguous().float() if g_per_scale is not None else None
        gt = g_total.contiguous().float() if g_total is not None else None
        g = torch.empty(2, S, device=ctx.weight.device, dtype=torch.float32)
        be.call("loss_combine_backward", S, C.c_void_p(_lib.ptr(gt)), C.c_void_p(_lib.ptr(gps)),
                C.c_void_p(ctx.weight.data_ptr()), C.c_float(ctx.num_scales), C.c_void_p(g.data_ptr()),
                C.c_void_p(g.data_ptr() + 4 * S))
        return g[0], g[1], None, None, None


def combine_losses(reproj, smooth, weight, num_scales, backend: Optional[_lib.Backend] = None):
    """``per_scale[s] = reproj[s] + weight[s] * smooth[s]``, ``total = sum(per_scale) / num_scales``."""
    be = backend if backend is not None else _lib.cuda_backend()
    return _Combine.apply(reproj, smooth, weight, num_scales, be)


class _PosePack(torch.autograd.Function):
    """T (n_pose,4,4) -> P = (K[k_row] @ T)[:, :3, :] with ATen-bmm rounding; gradient to T."""

    @staticmethod
    def forward(ctx, T, K, k_row, be):
        Tc, Kc = T.detach().contiguous(), K.detach().contiguous()
        be.check_device(Tc, Kc, k_row)
        n = Tc.shape[0]
        P = torch.empty(n, 3, 4, device=T.device, dtype=torch.float32)
        be.call("pose_pack_forward", n, C.c_void_p(Kc.data_ptr()), C.c_void_p(k_row.data_ptr()),
                C.c_void_p(Tc.data_ptr()), C.c_void_p(P.data_ptr()))
        ctx.save_for_backward(Kc, k_row)
        ctx.be = be
        return P

    @staticmethod
    def backward(ctx, gP):
        Kc, k_row = ctx.saved_tensors
        g = gP.contiguous()
        n = g.shape[0]
        gT = torch.empty(n, 4, 4, device=g.device, dtype=torch.float32)
        ctx.be.call("pose_pack_backward", n, C.c_void_p(Kc.data_ptr()), C.c_void_p(k_row.data_ptr()),
                    C.c_void_p(g.data_ptr()), C.c_void_p(gT.data_ptr()))
        return gT, None, None, None


def pack_poses(plan: LossPlan, K: torch.Tensor, T: Dict, T_err: Optional[Dict] = None,
               backend: Optional[_lib.Backend] = None) -> torch.Tensor:
    """Pack ``P = (K[:n] @ T_f)[:, :3, :]`` of every frame in ``plan.pose_slices()`` order.

    ``K[:n]`` (first n rows, not the selected samples' rows) is what the reference pairs
    with a frame's poses (``trainer.py:431``, ``layers.py:182``).  One concatenation and one
    tiny kernel whose elements follow the k-sequential FMA chain of ATen's bmm.
    """
    be = backend if backend is not None else _lib.cuda_backend()
    rows = []
    for f, is_err, lo, hi in plan.pose_slices():
        Tf = (T_err if is_err else T)[f]
        assert Tf.shape[0] == hi - lo, (f, Tf.shape, hi - lo)
        rows.append(Tf)
    if not rows:
        return K.new_zeros(0, 3, 4)
    T_all = torch.cat(rows, 0)
    cache = getattr(plan, "_k_rows", None)
    if cache is None or cache[0] != str(K.device):
        idx = [i for f, is_err, lo, hi in plan.pose_slices() for i in range(hi - lo)]
        cache = (str(K.device), torch.tensor(idx, dtype=torch.int32, device=K.device))
        plan._k_rows = cache
    if T_all.shape[0] == 0:
        return K.new_zeros(0, 3, 4)
    return _PosePack.apply(T_all, K, cache[1], be)
