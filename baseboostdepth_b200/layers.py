"""Drop-in for the reference's ``layers`` module (tier A: ``trainer.py`` runs unchanged).

``from baseboostdepth_b200.layers import SSIM, BackprojectDepth, Project3D,
transformation_from_parameters, disp_to_depth, get_smooth_loss, compute_depth_errors``
gives the names ``trainer.py:21-22`` imports; ``ConvBlock``, ``Conv3x3`` and ``upsample``
cover ``networks/depth_decoder.py:8``.  The four hot-path layers keep the reference's
constructor and ``forward`` signatures (``layers.py:136-249``) but run as
``torch.autograd.Function`` wrappers over ``libbbd_loss.so``; there is no CPU path.

This tier cannot fuse across the calls the trainer makes itself (``F.grid_sample``,
``torch.cat``/``min``, ``randn``): it exists for compatibility and for per-operator parity
tests.  The performance path is ``baseboostdepth_b200.trainer.FusedLossMixin``.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .geometry import (Conv3x3, ConvBlock, compute_depth_errors, disp_to_depth,  # noqa: F401  (re-exported)
                       get_translation_matrix, rot_from_axisangle, upsample)

_TEST_BACKEND = None  # tests/ may point this at the CPU emulation harness; the package never does


def _backend():
    return _TEST_BACKEND if _TEST_BACKEND is not None else _lib.cuda_backend()


def _p(t):
    return C.c_void_p(t.data_ptr() if t is not None else None)


class _Pose(torch.autograd.Function):
    @staticmethod
    def forward(ctx, axisangle, translation, invert):
        be = _backend()
        aa = axisangle.detach().reshape(-1, 3).contiguous()
        tr = translation.detach().reshape(-1, 3).contiguous()
        be.check_device(aa, tr)
        n = aa.shape[0]
        T = torch.empty(n, 4, 4, device=aa.device, dtype=torch.float32)
        be.call("pose_forward", n, _p(aa), _p(tr), int(invert), _p(T))
        ctx.save_for_backward(aa, tr)
        ctx.meta = (bool(invert), axisangle.shape, translation.shape)
        return T

    @staticmethod
    def backward(ctx, gT):
        be = _backend()
        aa, tr = ctx.saved_tensors
        invert, sa, st = ctx.meta
        g = gT.contiguous()
        gaa, gtr = torch.empty_like(aa), torch.empty_like(tr)
        be.call("pose_backward", aa.shape[0], _p(aa), _p(tr), int(invert), _p(g), _p(gaa), _p(gtr))
        return gaa.view(sa), gtr.view(st), None


def transformation_from_parameters(axisangle, translation, invert=False):
    """Network outputs ``(B,1,3)`` axis-angle and translation -> camera motion ``(B,4,4)``.

    Reference ``layers.py:25-42`` (with ``rot_from_axisangle`` ``:61-100`` and
    ``get_translation_matrix`` ``:45-58``): about forty tiny tensor kernels per call there, one
    kernel forward and one backward here.  The plain tensor version stays available as
    ``baseboostdepth_b200.geometry.transformation_from_parameters``.
    """
    return _Pose.apply(axisangle, translation, bool(invert))


class _Backproject(torch.autograd.Function):
    @staticmethod
    def forward(ctx, depth, inv_K, height, width):
        be = _backend()
        n = len(inv_K)
        depth_c = depth.detach().reshape(n, height * width).contiguous()
        ik = inv_K.detach().contiguous()
        be.check_device(depth_c, ik)
        points = torch.empty(n, 4, height * width, device=depth.device, dtype=torch.float32)
        be.call("backproject_forward", n, height, width, _p(depth_c), _p(ik), _p(points))
        ctx.save_for_backward(ik)
        ctx.shape = (depth.shape, height, width)
        return points

    @staticmethod
    def backward(ctx, gpoints):
        be = _backend()
        (ik,) = ctx.saved_tensors
        shape, height, width = ctx.shape
        n = ik.shape[0]
        g = gpoints.contiguous()
        gdepth = torch.empty(n, height * width, device=g.device, dtype=torch.float32)
        be.call("backproject_backward", n, height, width, _p(ik), _p(g), _p(gdepth))
        return gdepth.view(shape), None, None, None


class BackprojectDepth(nn.Module):
    """Depth image -> homogeneous camera points ``(n, 4, H*W)``.  Reference ``layers.py:136-167``.

    The reference precomputes a ``(batch, 3, H*W)`` pixel grid and a ones plane as frozen
    parameters (17.7 MB at 640x192, batch 12); the kernel derives both from the thread index,
    so this module has no state.  ``n = len(inv_K)`` may be smaller than ``batch_size``.
    Gradient flows to ``depth`` only (intrinsics carry no gradient in the trainer).
    """

    def __init__(self, batch_size, height, width):
        super().__init__()
        self.batch_size, self.height, self.width = batch_size, height, width

    def forward(self, depth, inv_K):
        if inv_K.requires_grad:
            raise NotImplementedError("bbd BackprojectDepth: gradient w.r.t. inv_K is not provided")
        return _Backproject.apply(depth, inv_K, self.height, self.width)


class _Project(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, P, height, width, eps):
        be = _backend()
        n = P.shape[0]
        pts = points.detach().contiguous()
        Pc = P.detach().contiguous()
        be.check_device(pts, Pc)
        pix = torch.empty(n, 2, height, width, device=points.device, dtype=torch.float32)
        be.call("project_forward", n, height, width, _p(pts), _p(Pc), C.c_float(eps), _p(pix))
        ctx.save_for_backward(pts, Pc)
        ctx.dims = (height, width, eps)
        # the reference returns the (n,H,W,2) permuted view of an (n,2,H,W) buffer (layers.py:189-190)
        return pix.permute(0, 2, 3, 1)

    @staticmethod
    def backward(ctx, gpix):
        be = _backend()
        pts, Pc = ctx.saved_tensors
        height, width, eps = ctx.dims
        n = Pc.shape[0]
        g = gpix.permute(0, 3, 1, 2).contiguous()
        gpoints = torch.empty_like(pts)
        chunks = be.value("project_chunks", height, width)
        gP_part = torch.empty(n, chunks, 12, device=pts.device, dtype=torch.float32)
        be.call("project_backward", n, height, width, _p(pts), _p(Pc), C.c_float(eps), _p(g), _p(gpoints), _p(gP_part))
        return gpoints, gP_part.sum(1).view(n, 3, 4), None, None, None


class Project3D(nn.Module):
    """Camera points -> sampling grid in [-1, 1], ``(n, H, W, 2)``.  Reference ``layers.py:170-195``."""

    def __init__(self, batch_size, height, width, eps=1e-7):
        super().__init__()
        self.batch_size, self.height, self.width, self.eps = batch_size, height, width, eps

    def forward(self, points, K, T):
        P = torch.matmul(K, T)[:, :3, :]          # tiny batched 4x4 product, kept in torch (autograd to T)
        return _Project.apply(points, P, self.height, self.width, float(self.eps))


class _SSIM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y):
        be = _backend()
        xc, yc = x.detach().contiguous(), y.detach().contiguous()
        be.check_device(xc, yc)
        n, c, h, w = xc.shape
        out = torch.empty_like(xc)
        be.call("ssim_forward", n, c, h, w, _p(xc), _p(yc), _p(out))
        ctx.save_for_backward(xc, yc)
        return out

    @staticmethod
    def backward(ctx, gout):
        be = _backend()
        xc, yc = ctx.saved_tensors
        n, c, h, w = xc.shape
        g = gout.contiguous()
        gx = torch.empty_like(xc) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(yc) if ctx.needs_input_grad[1] else None
        be.call("ssim_backward", n, c, h, w, _p(xc), _p(yc), _p(g), _p(gx), _p(gy))
        return gx, gy


class SSIM(nn.Module):
    """SSIM dissimilarity ``clamp((1 - SSIM)/2, 0, 1)`` with 3x3 reflection-padded mean pools.

    Reference ``layers.py:219-249``.  One kernel forward, one backward (window statistics are
    recomputed, nothing but ``x`` and ``y`` is saved -- the reference's autograd graph keeps
    ~25 full-size intermediates).
    """

    def __init__(self):
        super().__init__()
        self.C1, self.C2 = 0.01 ** 2, 0.03 ** 2

    def forward(self, x, y):
        return _SSIM.apply(x, y)


class _Smooth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, img):
        be = _backend()
        d, im = disp.detach().contiguous(), img.detach().contiguous()
        be.check_device(d, im)
        B, _, h, w = d.shape
        sa = _lib.SmoothArgs()
        sa.batch, sa.levels, sa.normalize = B, 1, 0
        sa.h[0], sa.w[0] = h, w
        sa.disp[0], sa.img[0] = d.data_ptr(), im.data_ptr()
        gdisp = torch.empty_like(d)
        sa.gdisp[0] = gdisp.data_ptr()
        hs, ws = (C.c_int32 * 1)(h), (C.c_int32 * 1)(w)
        scratch = torch.empty(max(1, be.value("smooth_scratch_floats", B, 1, hs, ws)), device=d.device,
                              dtype=torch.float32)
        loss = torch.empty(1, device=d.device, dtype=torch.float32)
        sa.scratch, sa.loss = scratch.data_ptr(), loss.data_ptr()
        be.call("smooth_fused", C.byref(sa))
        ctx.save_for_backward(gdisp, d, im)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        gdisp, d, im = ctx.saved_tensors
        gimg = None
        if ctx.needs_input_grad[1]:
            be = _backend()
            B, _, h, w = d.shape
            gs = g.detach().reshape(1).contiguous().float()
            gimg = torch.empty_like(im)
            ia = _lib.SmoothImgArgs()
            ia.batch, ia.levels = B, 1
            ia.h[0], ia.w[0] = h, w
            ia.disp[0], ia.img[0], ia.gimg[0] = d.data_ptr(), im.data_ptr(), gimg.data_ptr()
            ia.coef, ia.gscale = None, gs.data_ptr()     # no normalisation: r = 1
            be.call("smooth_image_grad", C.byref(ia))
        return gdisp * g, gimg


def get_smooth_loss(disp, img):
    """Edge-aware smoothness of a disparity image, 0-d tensor.  Reference ``layers.py:203-216``.

    One fused forward+backward pass (the gradient w.r.t. ``disp`` is produced with the value).
    When ``img`` requires grad, the backward adds one gather kernel for its gradient.  The trainer
    passes the mean-normalised disparity (``trainer.py:560-563``); the fused path folds that
    normalisation into the same kernel (``normalize=1``).
    """
    return _Smooth.apply(disp, img)


class _GridSample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, images, grid):
        be = _backend()
        img = images.detach().contiguous()
        g = grid.detach().permute(0, 3, 1, 2).contiguous()     # (n,2,Ho,Wo): no copy for Project3D's output
        be.check_device(img, g)
        n, c, h, w = img.shape
        ho, wo = g.shape[2], g.shape[3]
        out = torch.empty(n, c, ho, wo, device=img.device, dtype=torch.float32)
        be.call("grid_sample_forward", n, c, h, w, ho, wo, _p(img), _p(g), _p(out))
        ctx.save_for_backward(img, g)
        return out

    @staticmethod
    def backward(ctx, gout):
        be = _backend()
        img, g = ctx.saved_tensors
        n, c, h, w = img.shape
        ho, wo = g.shape[2], g.shape[3]
        go = gout.contiguous()
        gimg = gg = None
        if ctx.needs_input_grad[1]:
            gg = torch.empty_like(g)
            be.call("grid_sample_backward", n, c, h, w, ho, wo, _p(img), _p(g), _p(go), _p(gg))
            gg = gg.permute(0, 2, 3, 1)
        if ctx.needs_input_grad[0]:
            # transpose of the gather, sorted by destination (no atomics; the trainer itself never asks for it)
            keys = torch.empty(n * ho * wo, device=img.device, dtype=torch.int32)
            be.call("grid_sample_dest_keys", n, h, w, ho, wo, _p(g), _p(keys))
            keys_sorted, order = torch.sort(keys, stable=True)
            order = order.to(torch.int32)
            seg = torch.empty(n * h * w + 1, device=img.device, dtype=torch.int32)
            gimg = torch.empty_like(img)
            be.call("grid_sample_backward_image", n, c, h, w, ho, wo, _p(g), _p(go), _p(keys_sorted), _p(order), _p(seg), _p(gimg))
        return gimg, gg


def grid_sample(images, grid, align_corners=True, padding_mode="border", mode="bilinear"):
    """``F.grid_sample`` for the one configuration the trainer uses (``trainer.py:439,442``):
    bilinear, border padding, ``align_corners=True``.  Gradients flow to ``grid`` and, when asked for, to
    ``images`` (a deterministic sorted gather instead of ATen's atomic scatter).
    ``torch.nn.functional.grid_sample = baseboostdepth_b200.layers.grid_sample`` lets an unchanged
    ``trainer.py`` use it (tier A)."""
    if not (align_corners and padding_mode == "border" and mode == "bilinear"):
        raise NotImplementedError("bbd grid_sample implements bilinear / border / align_corners=True only")
    return _GridSample.apply(images, grid)
