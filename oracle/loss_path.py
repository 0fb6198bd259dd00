"""Oracle: the reference view-synthesis loss restated with host PyTorch ops.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

Every function follows the cited lines of ``/root/reference`` and issues the
same ATen ops in the same order, so on a given device its results equal the
reference's (checked bit-for-bit against ``tests/golden/*.npz``).  It works in
any floating dtype; the float64 run is the yardstick for fp32 tolerances.

Data layout follows the reference trainer: ``inputs[("color", f, s)]``,
``inputs[("K", 0)]``, ``inputs[("inv_K", 0)]``, ``inputs["stereo_T"]``,
``inputs["ordering"]``; ``outputs[("disp", s)]``, ``outputs[("cam_T_cam", 0, f)]``
(and ``("cam_T_cam_error", 0, f)`` for the error-induced variant).
"""
from __future__ import annotations

import re
from types import SimpleNamespace

import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------
# layers.py
# --------------------------------------------------------------------------
def pixel_grid(n, height, width, device, dtype):
    """Homogeneous pixel coordinates (n,3,HW): x fastest.  ``layers.py:139-158``."""
    ys, xs = torch.meshgrid(torch.arange(height, device=device, dtype=dtype),
                            torch.arange(width, device=device, dtype=dtype), indexing="ij")
    pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(height * width, device=device, dtype=dtype)], 0)
    return pix.unsqueeze(0).repeat(n, 1, 1)


def backproject(depth, inv_K, height, width):
    """Depth -> camera points (n,4,HW).  ``BackprojectDepth.forward`` ``layers.py:160-167``."""
    n = len(inv_K)
    pix = pixel_grid(n, height, width, depth.device, depth.dtype)
    cam = torch.matmul(inv_K[:, :3, :3], pix)
    cam = depth.view(n, 1, -1) * cam
    ones = torch.ones(n, 1, height * width, device=depth.device, dtype=depth.dtype)
    return torch.cat([cam, ones], 1)


def project(points, K, T, height, width, eps=1e-7):
    """Camera points -> sampling grid in [-1,1] (n,H,W,2).  ``Project3D.forward`` ``layers.py:181-195``."""
    P = torch.matmul(K, T)[:, :3, :]
    cam = torch.matmul(P, points)
    pix = cam[:, :2, :] / (cam[:, 2, :].unsqueeze(1) + eps)
    pix = pix.view(len(K), 2, height, width).permute(0, 2, 3, 1)
    pix[..., 0] /= width - 1
    pix[..., 1] /= height - 1
    return (pix - 0.5) * 2


def warp(images, grid):
    """Bilinear, border-padded, align_corners warp.  ``trainer.py:442`` (and ``:439``)."""
    return F.grid_sample(images, grid, align_corners=True, padding_mode="border")


def ssim(x, y):
    """SSIM dissimilarity map (n,3,H,W).  ``SSIM.forward`` ``layers.py:235-249``."""
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    x = F.pad(x, (1, 1, 1, 1), mode="reflect")
    y = F.pad(y, (1, 1, 1, 1), mode="reflect")
    mu_x = F.avg_pool2d(x, 3, 1)
    mu_y = F.avg_pool2d(y, 3, 1)
    sigma_x = F.avg_pool2d(x ** 2, 3, 1) - mu_x ** 2
    sigma_y = F.avg_pool2d(y ** 2, 3, 1) - mu_y ** 2
    sigma_xy = F.avg_pool2d(x * y, 3, 1) - mu_x * mu_y
    num = (2 * mu_x * mu_y + c1) * (2 * sigma_xy + c2)
    den = (mu_x ** 2 + mu_y ** 2 + c1) * (sigma_x + sigma_y + c2)
    return torch.clamp((1 - num / den) / 2, 0, 1)


def reprojection_loss(pred, target, no_ssim=False):
    """0.85*SSIM + 0.15*L1, channel-averaged (n,1,H,W).  ``trainer.py:477-486``."""
    l1 = torch.abs(target - pred).mean(1, True)
    if no_ssim:
        return l1
    return 0.85 * ssim(pred, target).mean(1, True) + 0.15 * l1


def smooth_loss(disp, img):
    """Edge-aware first-order smoothness.  ``get_smooth_loss`` ``layers.py:203-216``."""
    ddx = torch.abs(disp[:, :, :, :-1] - disp[:, :, :, 1:])
    ddy = torch.abs(disp[:, :, :-1, :] - disp[:, :, 1:, :])
    idx = torch.mean(torch.abs(img[:, :, :, :-1] - img[:, :, :, 1:]), 1, keepdim=True)
    idy = torch.mean(torch.abs(img[:, :, :-1, :] - img[:, :, 1:, :]), 1, keepdim=True)
    ddx = ddx * torch.exp(-idx)
    ddy = ddy * torch.exp(-idy)
    return ddx.mean() + ddy.mean()


def disp_to_depth(disp, min_depth, max_depth):
    """``layers.py:13-22``."""
    min_disp, max_disp = 1 / max_depth, 1 / min_depth
    scaled = min_disp + (max_disp - min_disp) * disp
    return scaled, 1 / scaled


def rot_from_axisangle(vec):
    """Axis-angle (n,1,3) -> homogeneous rotation (n,4,4), written element by element into zeros.
    ``layers.py:61-100``."""
    angle = torch.norm(vec, 2, 2, True)
    axis = vec / (angle + 1e-7)
    ca, sa = torch.cos(angle), torch.sin(angle)
    C = 1 - ca
    x, y, z = axis[..., 0].unsqueeze(1), axis[..., 1].unsqueeze(1), axis[..., 2].unsqueeze(1)
    xs, ys, zs = x * sa, y * sa, z * sa
    xC, yC, zC = x * C, y * C, z * C
    xyC, yzC, zxC = x * yC, y * zC, z * xC
    rot = torch.zeros((vec.shape[0], 4, 4), device=vec.device, dtype=vec.dtype)
    rot[:, 0, 0] = torch.squeeze(x * xC + ca)
    rot[:, 0, 1] = torch.squeeze(xyC - zs)
    rot[:, 0, 2] = torch.squeeze(zxC + ys)
    rot[:, 1, 0] = torch.squeeze(xyC + zs)
    rot[:, 1, 1] = torch.squeeze(y * yC + ca)
    rot[:, 1, 2] = torch.squeeze(yzC - xs)
    rot[:, 2, 0] = torch.squeeze(zxC - ys)
    rot[:, 2, 1] = torch.squeeze(yzC + xs)
    rot[:, 2, 2] = torch.squeeze(z * zC + ca)
    rot[:, 3, 3] = 1
    return rot


def get_translation_matrix(translation_vector):
    """Translation (n,1,3) -> homogeneous (n,4,4).  ``layers.py:45-58``."""
    T = torch.zeros(translation_vector.shape[0], 4, 4, device=translation_vector.device, dtype=translation_vector.dtype)
    t = translation_vector.contiguous().view(-1, 3, 1)
    for i in range(4):
        T[:, i, i] = 1
    T[:, :3, 3, None] = t
    return T


def transformation_from_parameters(axisangle, translation, invert=False):
    """(axis-angle, translation) -> 4x4 camera motion.  ``layers.py:25-42``."""
    R = rot_from_axisangle(axisangle)
    t = translation.clone()
    if invert:
        R = R.transpose(1, 2)
        t *= -1
    T = get_translation_matrix(t)
    return torch.matmul(R, T) if invert else torch.matmul(T, R)


# --------------------------------------------------------------------------
# trainer.py: sub-batch masks
# --------------------------------------------------------------------------
def initial_valid_frames(ordering):
    """``trainer.py:292`` -- deterministic order instead of ``list(set(...))``."""
    seen = []
    for entry in ordering:
        for el in entry:
            if el != 0 and el not in seen:
                seen.append(el)
    return sorted(seen, key=lambda f: (1 << 30) if f == "s" else 2 * abs(f) + (f < 0))


def frame_ids_from_ordering(ordering):
    """``custom_collate`` ``trainer.py:869-877`` + the abs-sort of ``:245-250``."""
    ms = [0 if o[1] == "s" else o[1] for o in ordering]
    top = max(ms)
    if top == 0:
        ids = [0, "s"]
    else:
        ids = list(range(-top, top + 1))
        if any(m in (0, 1, 2) for m in ms):
            ids.append("s")
    return sorted(ids, key=lambda f: float("inf") if isinstance(f, str) else abs(f))


def sub_batch_masks(ordering, frame_ids, valid_frames, trimin):
    """Boolean-list masks of ``Trainer.valid_frames_trimin`` ``trainer.py:888-981``.

    Returns a namespace with ``valid_mask_dict``, ``valid_mask`` and, for
    tri-min, ``valid_tri_mask_dict``, ``valid_tri_mask``,
    ``valid_tri_mask_reverse`` plus the extended ``valid_frames`` list.
    """
    base = [o[1] for o in ordering]
    vf = list(valid_frames)
    m = SimpleNamespace(valid_mask_dict={}, valid_mask={}, valid_tri_mask_dict={},
                        valid_tri_mask={}, valid_tri_mask_reverse={}, valid_frames=vf)

    def extend():
        # trainer.py:961-981
        if (1 in vf or 2 in vf) and "s" not in vf:
            vf.append("s")
        for low in range(1, 7):
            need = (low + 1 in vf or low + 2 in vf) if low < 6 else (7 in vf)
            if need and low not in vf:
                vf.extend([low, -low])

    for pos, f in enumerate(frame_ids[1:]):
        if "s" in vf and pos == 0:
            m.valid_mask_dict["s"] = [b == "s" for b in base]
        elif "s" not in vf:
            m.valid_mask_dict["s"] = [False for _ in base]
        if f != "s" and f > 0:
            m.valid_mask_dict[f] = [(b == f) if b != "s" else False for b in base]
            m.valid_mask[f] = [b == f for b in base if b != "s" and b >= f]

    if not trimin:
        return m

    rev = m.valid_tri_mask_reverse
    for pos, f in enumerate(frame_ids[1:]):
        if pos == 0:
            if "s" in vf or 1 in vf or 2 in vf:
                m.valid_tri_mask_dict["s"] = [b in ("s", 1, 2) for b in base]
            else:
                m.valid_tri_mask_dict["s"] = [False for _ in base]
        if f != "s" and f > 0:
            span = (f, f + 1, f + 2)
            m.valid_tri_mask_dict[f] = [(b in span) if b != "s" else False for b in base]
            m.valid_tri_mask[f] = [b in span for b in base if b != "s" and b >= f]
            if f < 6:
                rows = [b for b in base if b != "s" and f <= b <= f + 2]
                reach = (f, f + 1, f + 2)
            elif f == 6:
                rows = [b for b in base if b != "s" and b >= f]
                reach = (f, f + 1)
            else:  # f == 7
                rows = [b for b in base if b == f]
                reach = ()
                rev[f" {f}"] = [True for _ in rows]
                rev[f"{-f}"] = rev[f" {f}"]
            for g in reach:
                if g in vf:
                    tag = f"{f}" if g == f else f"{f}+{g}"
                    rev[" " + tag] = [b == g for b in rows]
            for g in reach:
                if g in vf:
                    tag = f"{-f}" if g == f else f"{-f}+{g}"
                    src = f" {f}" if g == f else f" {f}+{g}"
                    rev[tag] = rev[src]
        elif f == "s":
            rows = [b for b in base if b == "s" or b <= 2]
            if "s" in vf:
                rev["s"] = [b == "s" for b in rows]
            for g in (1, 2):
                if g in vf:
                    rev[f"s+{g}"] = [b == g for b in rows]
    extend()  # once, after the masks are built (trainer.py:961 sits outside both loops)
    return m


def _pick(t, mask):
    return t[mask]


# --------------------------------------------------------------------------
# trainer.py: view synthesis
# --------------------------------------------------------------------------
def view_synthesis(inputs, outputs, opt, masks):
    """``Trainer.generate_images_pred`` + ``warping_block_for_easy_looking`` ``trainer.py:421-475``.

    Fills ``outputs[("depth",0,s)]``, ``outputs[("color",f,s)]`` and, with
    ``opt.decomp``, ``outputs[("color_D",f,s)]``; also records the sampling
    grids under ``outputs[("grid",f,s)]`` for coordinate parity checks.
    """
    sel_rows = masks.valid_tri_mask if opt.trimin else masks.valid_mask
    sel_batch = masks.valid_tri_mask_dict if opt.trimin else masks.valid_mask_dict
    H, W = opt.height, opt.width
    for s in opt.scales:
        disp = F.interpolate(outputs[("disp", s)], [H, W], mode="bilinear", align_corners=False)
        depth = disp if opt.SQL else disp_to_depth(disp, opt.min_depth, opt.max_depth)[1]
        outputs[("depth", 0, s)] = depth
        for f in masks.valid_frames:
            if f == "s":
                T = _pick(inputs["stereo_T"], sel_batch["s"])
                T_err = None
                images = inputs[("color", "s", 0)]
                d = _pick(depth, sel_batch["s"])
            else:
                T = outputs[("cam_T_cam", 0, f)]
                T_err = outputs[("cam_T_cam_error", 0, f)] if opt.decomp else None
                images = _pick(inputs[("color", f, 0)], sel_rows[abs(f)])
                d = _pick(depth, sel_batch[abs(f)])
            n = T.shape[0]
            K = inputs[("K", 0)][:n]
            inv_K = inputs[("inv_K", 0)][:n]
            cam = backproject(d, inv_K, H, W)
            if opt.decomp and f != "s":
                grid_err = project(cam, K, T_err, H, W)
                outputs[("color_D", f, s)] = warp(images, grid_err)
                outputs[("grid_D", f, s)] = grid_err
            grid = project(cam, K, T, H, W)
            outputs[("grid", f, s)] = grid
            outputs[("color", f, s)] = warp(images, grid)
    return outputs


# --------------------------------------------------------------------------
# trainer.py: losses
# --------------------------------------------------------------------------
_NUM = re.compile(r"-?\d+")


def group_order(ordering, masks, trimin):
    """Groups in the order noise is drawn (``temp_positive``, ``trainer.py:516-523``)."""
    src = initial_valid_frames(ordering) if trimin else masks.valid_frames
    return [f for f in src if f == "s" or f > 0]


def _tri_keys(g):
    """Candidate keys of group g in ``Trainer.x_min_opt`` order (``trainer.py:983-1100``)."""
    if g == "s":
        return ["s"]
    if g == 1:
        return ["1", "-1", "s+1"]
    if g == 2:
        return ["2", "-2", "1+2", "-1+2", "s+2"]
    return [f"{g}", f"{-g}", f"{g-1}+{g}", f"{-g+1}+{g}", f"{g-2}+{g}", f"{-g+2}+{g}"]


def _rekey(per_frame, rev, skip_stereo=False):
    """``trainer.py:513-515,536-540``: split per-frame planes into per-(source, group) planes."""
    out = {}
    for key, mask in rev.items():
        name = key[1:] if key[0] == " " else key
        if key[0] == "s":
            if skip_stereo:
                continue
            out[name] = per_frame["s"][mask]
        else:
            out[name] = per_frame[int(_NUM.search(key).group())][mask]
    return out


def losses(inputs, outputs, opt, masks, noise, num_scales=None):
    """``Trainer.compute_losses`` ``trainer.py:488-570`` with explicit ``noise``.

    ``noise[g]`` is the already scaled (``randn * 1e-5``) plane stack of group
    g (``trainer.py:518,522``).  Returns ``(losses, aux)`` where ``aux`` holds,
    per scale, the per-group minima ``to_optimise`` and ``argmin`` planes.
    """
    frames = masks.valid_frames
    sel_rows = masks.valid_tri_mask if opt.trimin else masks.valid_mask
    sel_batch = masks.valid_tri_mask_dict if opt.trimin else masks.valid_mask_dict
    num_scales = num_scales if num_scales is not None else len(opt.scales)
    color0 = inputs[("color", 0, 0)]

    target = {f: color0[sel_batch[abs(f)] if f != "s" else sel_batch["s"]] for f in frames}
    source = {f: (inputs[("color", f, 0)][sel_rows[abs(f)]] if f != "s" else inputs[("color", "s", 0)])
              for f in frames}
    ident = {f: reprojection_loss(source[f], target[f], opt.no_ssim) for f in frames}
    groups = group_order(inputs["ordering"], masks, opt.trimin)
    if opt.trimin:
        ident = _rekey(ident, masks.valid_tri_mask_reverse)

    out, aux = {}, {"to_optimise": {}, "argmin": {}, "planes": {}, "groups": groups}
    total = 0
    for s in opt.scales:
        rep = {f: reprojection_loss(outputs[("color", f, s)], target[f], opt.no_ssim) for f in frames}
        rep_d = None
        if opt.decomp:
            rep_d = {f: reprojection_loss(outputs[("color_D", f, s)], target[f], opt.no_ssim)
                     for f in frames if f != "s"}
        if opt.trimin:
            rep = _rekey(rep, masks.valid_tri_mask_reverse)
            if opt.decomp:
                rep_d = _rekey(rep_d, masks.valid_tri_mask_reverse, skip_stereo=True)

        mins, args, cats = [], [], []
        for g in groups:
            if opt.trimin:
                keys = _tri_keys(g)
                planes = [rep[k] for k in keys]
                if opt.decomp:
                    planes += [rep_d[k] for k in keys if not k.startswith("s")]
                planes += [ident[k] + noise[g] for k in keys]
            elif g == "s":
                planes = [rep["s"], ident["s"] + noise["s"]]
            else:
                planes = [rep[g], rep[-g], ident[g] + noise[g], ident[-g] + noise[g]]
            stacked = torch.cat(planes, dim=1)
            val, idx = torch.min(stacked, dim=1)
            mins.append(val)
            args.append(idx)
            cats.append(stacked.detach())
        to_optimise = torch.cat(mins, dim=0)
        aux["to_optimise"][s] = mins
        aux["argmin"][s] = args
        aux["planes"][s] = cats

        loss = to_optimise.mean()
        disp = outputs[("disp", s)]
        color = inputs[("color", 0, s)]
        if color.shape[-2:] != disp.shape[-2:] and opt.SQL:
            disp = F.interpolate(disp, [opt.height, opt.width], mode="bilinear", align_corners=False)
        mean_disp = disp.mean(2, True).mean(3, True)
        norm_disp = disp / (mean_disp + 1e-7)
        loss = loss + opt.disparity_smoothness * smooth_loss(norm_disp, color) / (2 ** s)
        total = total + loss
        out[f"loss/{s}"] = loss
    out["loss"] = total / num_scales
    return out, aux


def default_opt(**kw):
    """Option namespace with the reference defaults that the loss path reads (``options.py``)."""
    opt = SimpleNamespace(height=192, width=640, scales=[0, 1, 2, 3], min_depth=0.1, max_depth=100.0,
                          disparity_smoothness=1e-3, no_ssim=False, trimin=False, decomp=False,
                          pose_error=1, SQL=False, incremental_skip=False, partial_skip=False,
                          batch_size=12, frame_ids=[0, -1, 1])
    for k, v in kw.items():
        setattr(opt, k, v)
    return opt


def run(inputs, outputs, opt, noise, num_scales=None):
    """Whole path: masks -> view synthesis -> losses.  Mirrors ``process_batch`` ``trainer.py:292-298``."""
    ordering = inputs["ordering"]
    frame_ids = frame_ids_from_ordering(ordering)
    masks = sub_batch_masks(ordering, frame_ids, initial_valid_frames(ordering), opt.trimin)
    view_synthesis(inputs, outputs, opt, masks)
    out, aux = losses(inputs, outputs, opt, masks, noise, num_scales)
    aux["masks"] = masks
    return out, aux
