"""Gradients of the fused loss w.r.t. the colour frames on the CUDA library vs the oracle (B200)."""
import pytest
import torch

from baseboostdepth_b200.synthetic import WORKLOADS, make_batch, make_noise
from baseboostdepth_b200.trainer import plan_for
from frame_grad_util import frame_grad, frame_keys, referenced_rows, require_frame_grads
from fused_util import mirror_to_device, run_fused
from helpers import PARITY_LOG, Golden, assert_grad_parity, golden_cases, near_tie_mask, rel_l2
from oracle import loss_path as O

pytestmark = pytest.mark.gpu


def _to_gpu(inputs, outputs, params, device, keys):
    gi, go, leaves = mirror_to_device(inputs, outputs, params, device)
    for k in keys:
        gi[k] = inputs[k].detach().to(device).requires_grad_(True)
    return gi, go, leaves


@pytest.mark.parametrize("case", golden_cases())
def test_golden_frame_grads_on_gpu(case, cuda_device):
    g = Golden(case)
    keys = frame_keys(g.inputs)
    require_frame_grads(g.inputs, keys)
    ref, aux = O.run(g.inputs, g.outputs, g.opt(), g.noise, num_scales=g.num_scales)
    ref["loss"].backward()
    h = Golden(case)
    gi, go, leaves = _to_gpu(h.inputs, h.outputs, h.params, cuda_device, keys)
    losses, plan = run_fused(gi, go, h.opt(), {k: v.to(cuda_device) for k, v in h.noise.items()}, h.num_scales,
                             groups=aux["groups"])
    losses["loss"].backward()
    torch.cuda.synchronize()
    for k, v in ref.items():
        assert abs(float(losses[k]) - float(v)) <= 2e-6 * max(1.0, abs(float(v))), k
    ref64, used = None, referenced_rows(plan)
    for k in keys:
        mine = frame_grad(gi, k).cpu()
        if rel_l2(mine, frame_grad(g.inputs, k)) > 1e-5 and ref64 is None:
            d = Golden(case, dtype=torch.float64)
            require_frame_grads(d.inputs, keys)
            O.run(d.inputs, d.outputs, d.opt(), d.noise, num_scales=d.num_scales)[0]["loss"].backward()
            ref64 = d
        assert_grad_parity(mine, frame_grad(g.inputs, k), None if ref64 is None else frame_grad(ref64.inputs, k), k,
                           case=case)
        if k[2] == 0 and k[1] != 0:
            for r in range(mine.shape[0]):
                if k[1] not in used or r not in used[k[1]]:
                    assert float(mine[r].abs().max()) == 0.0, (k, r)


def _source_footprint(plan, aux, outputs, masks, inputs, opt, f):
    """(rows,3,H,W) bool: bilinear taps (from the oracle's own sampling grids) of the 3x3 neighbourhoods of the
    1-dilated near-tie pixels, plus those pixels themselves (identity candidates read the row unwarped)."""
    stack = inputs[("color", f, 0)]
    rows, _, H, W = stack.shape
    out = torch.zeros(rows, H, W, dtype=torch.bool)
    sel_rows = masks.valid_tri_mask if opt.trimin else masks.valid_mask
    sel_batch = masks.valid_tri_mask_dict if opt.trimin else masks.valid_mask_dict
    if f == "s":
        row_idx, b_idx = list(range(rows)), [i for i, m in enumerate(sel_batch["s"]) if m]
    else:
        row_idx = [i for i, m in enumerate(sel_rows[abs(f)]) if m]
        b_idx = [i for i, m in enumerate(sel_batch[abs(f)]) if m]
    for s in opt.scales:
        near = near_tie_mask(plan, aux, s, dilate=2)
        for tag in ("grid", "grid_D"):
            grid = outputs.get((tag, f, s))
            if grid is None:
                continue
            grid = grid.detach()
            ix = ((grid[..., 0] + 1) / 2 * (W - 1)).clamp(0, W - 1).floor().long()
            iy = ((grid[..., 1] + 1) / 2 * (H - 1)).clamp(0, H - 1).floor().long()
            for i, (r, b) in enumerate(zip(row_idx, b_idx)):
                m = near[b]
                out[r] |= m
                xs, ys = ix[i][m], iy[i][m]
                for dy in (0, 1):
                    for dx in (0, 1):
                        out[r, (ys + dy).clamp(max=H - 1), (xs + dx).clamp(max=W - 1)] = True
    return out.unsqueeze(1).expand(rows, 3, H, W)


@pytest.mark.parametrize("name", ["kitti_640x192_b12_pm1", "trimin_decomp_640x192_b12"])
def test_full_size_frame_grads(name, cuda_device):
    batch, H, W, baselines, trimin, decomp = WORKLOADS[name]
    scales = [0, 1, 2, 3]
    opt = O.default_opt(height=H, width=W, trimin=trimin, decomp=decomp, pose_error=5.5, scales=scales, batch_size=batch)
    cfg = dict(batch=batch, height=H, width=W, baselines=list(baselines), trimin=trimin, decomp=decomp)
    inputs, outputs, params = make_batch(seed=1234, device="cpu", scales=scales, **cfg)
    keys = frame_keys(inputs)
    require_frame_grads(inputs, keys)
    plan = plan_for(inputs["ordering"], opt.trimin, opt.decomp,
                    inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
    noise = make_noise(plan, H, W, seed=4321)
    ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()

    fresh, fresh_out, fresh_params = make_batch(seed=1234, device="cpu", scales=scales, **cfg)
    gi, go, leaves = _to_gpu(fresh, fresh_out, fresh_params, cuda_device, keys)
    gnoise = {k: v.to(cuda_device) for k, v in noise.items()}
    losses, plan = run_fused(gi, go, opt, gnoise, 4, groups=aux["groups"])
    losses["loss"].backward()
    torch.cuda.synchronize()
    for k in ref:
        assert abs(float(losses[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), k

    ref64 = None
    near_any = torch.stack([near_tie_mask(plan, aux, s, dilate=1) for s in scales]).any(0)
    for k in keys:
        mine, want = frame_grad(gi, k).cpu(), frame_grad(inputs, k)
        if rel_l2(mine, want) > 1e-5 and ref64 is None:
            i64, o64, _ = make_batch(seed=1234, device="cpu", dtype=torch.float64, scales=scales, **cfg)
            require_frame_grads(i64, keys)
            O.run(i64, o64, opt, {kk: v.double() for kk, v in noise.items()}, num_scales=4)[0]["loss"].backward()
            ref64 = i64
        assert_grad_parity(mine, want, None if ref64 is None else frame_grad(ref64, k), k, case=name)
        if k[2] != 0 or not mine.numel():
            continue
        if k[1] == 0:
            foot = near_any.unsqueeze(1).expand_as(mine)
        else:
            foot = _source_footprint(plan, aux, outputs, aux["masks"], inputs, opt, k[1])
        off = (mine.double() - want.double()).abs() > 1e-5 * want.abs().max().item()
        frac_foot = foot.double().mean().item()
        frac_off = (off & ~foot).double().mean().item()
        PARITY_LOG.append({"case": name, "key": f"per-pixel d loss/d {k}", "footprint_fraction": frac_foot,
                           "pixels_off_by_1e-5_of_peak_outside_footprint": frac_off,
                           "pixels_off_anywhere": off.double().mean().item()})
        assert frac_off <= 1e-4, (k, frac_off)


def _step(case, device, frames_grad):
    h = Golden(case)
    keys = frame_keys(h.inputs)
    gi, go, leaves = _to_gpu(h.inputs, h.outputs, h.params, device, keys if frames_grad else [])
    calls = []
    from baseboostdepth_b200 import _lib
    be = _lib.cuda_backend()
    orig = be.call

    def rec(name, *args):
        calls.append(name)
        return orig(name, *args)

    be.call = rec
    try:
        losses, _ = run_fused(gi, go, h.opt(), {k: v.to(device) for k, v in h.noise.items()}, h.num_scales)
        losses["loss"].backward()
    finally:
        del be.call
    torch.cuda.synchronize()
    return losses, leaves, {k: frame_grad(gi, k).cpu() for k in keys} if frames_grad else None, calls


@pytest.mark.parametrize("case", ["plain_pm1", "trimin_decomp"])
def test_frame_grads_deterministic_and_default_path_unchanged(case, cuda_device):
    l1, leaves1, f1, c1 = _step(case, cuda_device, True)
    l2, leaves2, f2, c2 = _step(case, cuda_device, True)
    for k in f1:
        assert torch.equal(f1[k], f2[k]), k
    l0, leaves0, _, c0 = _step(case, cuda_device, False)
    assert not {"frame_grad", "frame_grad_stacks", "smooth_image_grad"} & set(c0), c0
    assert {"frame_grad", "frame_grad_stacks", "smooth_image_grad"} <= set(c1), c1
    for k in l0:
        assert torch.equal(l0[k].detach().cpu(), l1[k].detach().cpu()), k
    for k in leaves0:
        assert torch.equal(leaves0[k].grad.cpu(), leaves1[k].grad.cpu()), k
