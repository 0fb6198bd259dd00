"""Tier A -- the ``baseboostdepth_b200.layers`` drop-in that runs the reference's ``trainer.py`` unchanged -- against
the oracle, on the device, at the shapes where its launch code matters: chunked reductions with partial and
exactly-full chunks, grid-stride loops past the 148 x 16-block grid cap (606,208 threads at 256 per block, 303,104
for the SSIM gradient at 128), smoothness rows with several column blocks and the batch limit of 256, sub-batches
smaller than the module's batch size, and the edges of each operator (2-pixel images, coordinates on and outside
the border, zero rotations).

Bars.  Forward values: max |mine - fp32 ATen on the CPU| <= 1e-6.  Gradients: helpers.assert_grad_parity, i.e.
rel-L2 <= 1e-5 against the fp32 oracle (2e-5 for SSIM).  Where a bar is missed, the kernel may be no farther from
a float64 evaluation of the same op than fp32 ATen is.  On shapes of at most a few hundred pixels the float64
restatement in oracle/pixel_model.py is a second, torch-free yardstick.  Every comparison lands in PARITY_LOG.
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import baseboostdepth_b200.layers as L
from baseboostdepth_b200 import _lib
from baseboostdepth_b200.synthetic import WORKLOADS, make_batch, make_noise
from baseboostdepth_b200.trainer import plan_for
from frame_grad_util import frame_grad, frame_keys, require_frame_grads
from fused_util import mirror_to_device, retain_pose_grads
from helpers import PARITY_LOG, Golden, assert_grad_parity, golden_cases, max_abs, rel_l2
from oracle import loss_path as O
from oracle import pixel_model as PM

pytestmark = pytest.mark.gpu

GRID_CAP_THREADS = 148 * 16 * 256


def _sync(dev):
    if dev.type == "cuda":
        torch.cuda.synchronize()


def check_forward(mine, ref32, ref64, case, key, tol=1e-6):
    """max|mine - fp32 ATen| <= tol; where missed, no farther from float64 than fp32 ATen is (x2 + 1e-7)."""
    e = max_abs(mine, ref32)
    entry = {"case": case, "key": repr(key), "max_abs_vs_fp32_aten": e, "bar": "max_abs_vs_fp32_aten<=%g" % tol}
    ok = e <= tol
    if not ok and ref64 is not None:
        e_mine, e_ref = max_abs(mine, ref64), max_abs(ref32, ref64)
        entry.update(max_abs_vs_f64=e_mine, fp32_aten_vs_f64=e_ref, bar="no_farther_from_f64_than_fp32_aten(x2+1e-7)")
        ok = e_mine <= 2.0 * e_ref + 1e-7
        print(f"[parity] secondary bar for {case} {key}: vs fp32 ATen {e:.3e}, vs f64 {e_mine:.3e}, ATen vs f64 {e_ref:.3e}")
    entry["passed"] = bool(ok)
    PARITY_LOG.append(entry)
    assert ok, entry


def check_pixel_model(mine, aten32, model, case, key, grad=False):
    """Against the torch-free float64 restatement: no farther from it than fp32 ATen is.  Values: max-abs, x2 +
    5e-7; gradients: rel-L2, x2 + 2e-6 (assert_grad_parity's secondary bar)."""
    model = torch.as_tensor(np.asarray(model))
    metric = rel_l2 if grad else max_abs
    e_mine, e_ref = metric(mine, model), metric(aten32, model)
    ok = e_mine <= 2.0 * e_ref + (2e-6 if grad else 5e-7)
    PARITY_LOG.append({"case": case, "key": repr(key), "metric": metric.__name__, "vs_pixel_model_f64": e_mine,
                       "fp32_aten_vs_pixel_model_f64": e_ref, "bar": "no_farther_from_pixel_model_than_fp32_aten",
                       "passed": bool(ok)})
    assert ok, (case, key, e_mine, e_ref)


def _leaf(t, dev=None, dtype=None):
    return t.detach().to(device=dev if dev is not None else t.device, dtype=dtype or t.dtype).clone().requires_grad_(True)


# ------------------------------------------------------------------------------------------------------------------
# a. the reference trainer through tier A
# ------------------------------------------------------------------------------------------------------------------
def run_tier_a(monkeypatch, inputs, outputs, opt, noise, num_scales, batch_size):
    """oracle.loss_path -- the reference's generate_images_pred + compute_losses call for call -- with every layers.py
    operator it uses (and F.grid_sample) replaced by the drop-in, as an unchanged trainer.py would run."""
    with monkeypatch.context() as m:
        m.setattr(O, "backproject", lambda d, inv_K, H, W: L.BackprojectDepth(batch_size, H, W)(d, inv_K))
        m.setattr(O, "project", lambda cam, K, T, H, W: L.Project3D(batch_size, H, W)(cam, K, T))
        m.setattr(O, "warp", L.grid_sample)
        m.setattr(O, "ssim", L.SSIM())
        m.setattr(O, "smooth_loss", L.get_smooth_loss)
        m.setattr(O, "disp_to_depth", L.disp_to_depth)
        losses, _ = O.run(inputs, outputs, opt, noise, num_scales=num_scales)
        losses["loss"].backward()
    return losses


def _compare_losses(losses, ref, case):
    for k, v in ref.items():
        got, want = float(losses[k]), float(v)
        PARITY_LOG.append({"case": case, "key": repr(k), "loss": got, "oracle": want, "bar": "rel<=2e-6",
                           "passed": abs(got - want) <= 2e-6 * max(1.0, abs(want))})
        assert abs(got - want) <= 2e-6 * max(1.0, abs(want)), (case, k, got, want)


@pytest.mark.parametrize("frames", [False, True], ids=["frames_const", "frames_grad"])
@pytest.mark.parametrize("case", golden_cases())
def test_reference_trainer_through_tier_a(case, frames, cuda_device, monkeypatch):
    dev = cuda_device
    tag = f"tierA/{case}/{'frames' if frames else 'noframes'}"
    g = Golden(case)
    keys = frame_keys(g.inputs) if frames else []
    require_frame_grads(g.inputs, keys)
    retain_pose_grads(g.outputs)
    ref, _ = O.run(g.inputs, g.outputs, g.opt(), g.noise, num_scales=g.num_scales)
    ref["loss"].backward()
    g64 = Golden(case, dtype=torch.float64)
    require_frame_grads(g64.inputs, keys)
    retain_pose_grads(g64.outputs)
    O.run(g64.inputs, g64.outputs, g64.opt(), g64.noise, num_scales=g.num_scales)[0]["loss"].backward()

    h = Golden(case)
    gi, go, leaves = mirror_to_device(h.inputs, h.outputs, h.params, dev)
    for k in keys:
        gi[k] = _leaf(h.inputs[k], dev)
    noise = {k: v.to(dev) for k, v in h.noise.items()}
    losses = run_tier_a(monkeypatch, gi, go, h.opt(), noise, h.num_scales, len(h.baselines))
    _sync(dev)
    _compare_losses(losses, ref, tag)
    for k, leaf in leaves.items():
        ref32 = g.params[k].grad if k[0] == "disp" else g.outputs[k].grad
        r64 = g64.params[k].grad if k[0] == "disp" else g64.outputs[k].grad
        assert_grad_parity(leaf.grad, ref32, r64, k, case=tag)
    for k in keys:
        assert_grad_parity(frame_grad(gi, k).cpu(), frame_grad(g.inputs, k), frame_grad(g64.inputs, k), k, case=tag)


def test_reference_trainer_through_tier_a_full_size(cuda_device, monkeypatch):
    """The benchmark's batch: 30 projection chunks per sample, every tier-A grid above the cap."""
    name = "kitti_640x192_b12_pm1"
    batch, H, W, baselines, trimin, decomp = WORKLOADS[name]
    scales = [0, 1, 2, 3]
    opt = O.default_opt(height=H, width=W, trimin=trimin, decomp=decomp, pose_error=5.5, scales=scales, batch_size=batch)
    cfg = dict(batch=batch, height=H, width=W, baselines=list(baselines), trimin=trimin, decomp=decomp)
    inputs, outputs, params = make_batch(seed=1234, device="cpu", scales=scales, **cfg)
    plan = plan_for(inputs["ordering"], opt.trimin, opt.decomp, None)
    noise = make_noise(plan, H, W, seed=4321)
    retain_pose_grads(outputs)
    ref, _ = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()
    i64, o64, p64 = make_batch(seed=1234, device="cpu", dtype=torch.float64, scales=scales, **cfg)
    retain_pose_grads(o64)
    O.run(i64, o64, opt, {k: v.double() for k, v in noise.items()}, num_scales=4)[0]["loss"].backward()

    gi, go, leaves = mirror_to_device(inputs, outputs, params, cuda_device)
    losses = run_tier_a(monkeypatch, gi, go, opt, {k: v.to(cuda_device) for k, v in noise.items()}, 4, batch)
    _sync(cuda_device)
    tag = "tierA/" + name
    _compare_losses(losses, ref, tag)
    for k, leaf in leaves.items():
        ref32 = params[k].grad if k[0] == "disp" else outputs[k].grad
        r64 = p64[k].grad if k[0] == "disp" else o64[k].grad
        assert_grad_parity(leaf.grad, ref32, r64, k, case=tag)


# ------------------------------------------------------------------------------------------------------------------
# b. per-operator sweep
# ------------------------------------------------------------------------------------------------------------------
def _camera(n, H, W, gen):
    K = torch.tensor([[0.58 * W, 0, 0.5 * W, 0], [0, 1.92 * H, 0.5 * H, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]])
    K = K.unsqueeze(0).repeat(n, 1, 1)
    K[:, 0, 0] *= 1 + 0.1 * torch.rand(n, generator=gen)          # per-sample intrinsics
    return K, torch.linalg.pinv(K)


# 4095 / 4096 / 4097 / 4500 pixels: one partial chunk, one full chunk, a full chunk plus one pixel, two chunks;
# 192x640: 30 chunks and 12 x 122,880 pixels, past the grid cap.  9x13: small enough for the pixel model.
BP_SHAPES = [(63, 65), (64, 64), (17, 241), (50, 90), (192, 640), (9, 13)]


@pytest.mark.parametrize("n", [1, 3, 12])
@pytest.mark.parametrize("hw", BP_SHAPES, ids=[f"{h}x{w}" for h, w in BP_SHAPES])
def test_backproject_project_sweep(hw, n, cuda_device):
    dev = cuda_device
    H, W = hw
    case = f"backproject_project/{H}x{W}/n{n}"
    gen = torch.Generator().manual_seed(H * 1000 + W + n)
    K, inv_K = _camera(n + 2, H, W, gen)
    aa, tr = 0.05 * torch.randn(n, 1, 3, generator=gen), 0.1 * torch.randn(n, 1, 3, generator=gen)
    depth = 1 + 5 * torch.rand(n, 1, H, W, generator=gen)
    w = torch.rand(n, H, W, 2, generator=gen) + 0.5

    def chain(mods, d, a, t, Ks, iKs):
        T = mods[0](a, t)
        cam = mods[1](d, iKs)
        return T, cam, mods[2](cam, Ks, T)

    ours = (L.transformation_from_parameters, L.BackprojectDepth(n + 2, H, W), L.Project3D(n + 2, H, W))
    oracle = (O.transformation_from_parameters, lambda d, iK: O.backproject(d, iK, H, W),
              lambda cam, K_, T: O.project(cam, K_, T, H, W))
    d_g, a_g, t_g = _leaf(depth, dev), _leaf(aa, dev), _leaf(tr, dev)
    T_g, cam_g, grid_g = chain(ours, d_g, a_g, t_g, K[:n].to(dev), inv_K[:n].to(dev))   # batch_size > n
    (grid_g * w.to(dev)).sum().backward()
    _sync(dev)
    refs = {}
    for dt in (torch.float32, torch.float64):
        d, a, t = _leaf(depth, dtype=dt), _leaf(aa, dtype=dt), _leaf(tr, dtype=dt)
        T, cam, grid = chain(oracle, d, a, t, K[:n].to(dt), inv_K[:n].to(dt))
        (grid * w.to(dt)).sum().backward()
        # the same chain from the device's pose, so that the grid compares Project3D alone
        Td = T_g.detach().cpu().to(dt)
        refs[dt] = dict(T=T.detach(), cam=cam.detach(), grid=O.project(cam.detach(), K[:n].to(dt), Td, H, W), d=d.grad,
                        a=a.grad, t=t.grad)
    r32, r64 = refs[torch.float32], refs[torch.float64]
    check_forward(T_g, r32["T"], r64["T"], case, "T")
    check_forward(cam_g, r32["cam"], r64["cam"], case, "points")
    check_forward(grid_g, r32["grid"], r64["grid"], case, "grid")
    assert grid_g.shape == r32["grid"].shape and grid_g.stride() == (H * W * 2, W, 1, H * W)   # the reference's view
    assert_grad_parity(d_g.grad, r32["d"], r64["d"], "d/d depth", case=case)
    assert_grad_parity(a_g.grad, r32["a"], r64["a"], "d/d axisangle", case=case)
    assert_grad_parity(t_g.grad, r32["t"], r64["t"], "d/d translation", case=case)
    if H * W <= 300:
        Td = T_g.detach().cpu().double().numpy()
        model = np.stack([PM.backproject_project(depth[b, 0].double().numpy(), inv_K[b].double().numpy(),
                                                 K[b].double().numpy(), Td[b]) for b in range(n)])
        check_pixel_model(grid_g, r32["grid"], model, case, "grid")


SSIM_SHAPES = [(1, 1, 2, 2), (1, 3, 2, 7), (2, 3, 3, 5), (1, 4, 33, 57), (12, 3, 192, 640)]


@pytest.mark.parametrize("grads", ["x", "y", "xy"])
@pytest.mark.parametrize("shape", SSIM_SHAPES, ids=["x".join(map(str, s)) for s in SSIM_SHAPES])
def test_ssim_sweep(shape, grads, cuda_device):
    dev = cuda_device
    case = f"ssim/{'x'.join(map(str, shape))}/grad_{grads}"
    n, c, h, w = shape
    gen = torch.Generator().manual_seed(n * c * h * w + len(grads))
    x0, y0 = torch.rand(*shape, generator=gen), torch.rand(*shape, generator=gen)
    x0[..., 0, 0] = y0[..., 0, 0]          # a window of equal patches: dissimilarity near the clamp at 0
    up = torch.rand(*shape, generator=gen) - 0.25

    def run(x, y, fn):
        xg = x.detach().requires_grad_("x" in grads)
        yg = y.detach().requires_grad_("y" in grads)
        out = fn(xg, yg)
        (out * up.to(out.device, out.dtype)).sum().backward()
        return out.detach(), xg.grad, yg.grad

    # x non-contiguous on the device when both need a gradient: every other column of a wider buffer
    xd = x0.to(dev)
    if grads == "xy":
        xd = torch.zeros(n, c, h, 2 * w, device=dev)
        xd[..., ::2] = x0.to(dev)
        xd = xd[..., ::2]
    assert xd.is_contiguous() == (grads != "xy")
    mine = run(xd, y0.to(dev), L.SSIM())
    _sync(dev)
    r32 = run(x0.clone(), y0.clone(), O.ssim)
    r64 = run(x0.double(), y0.double(), O.ssim)
    check_forward(mine[0], r32[0], r64[0], case, "ssim")
    for i, name in ((1, "x"), (2, "y")):
        if name in grads:
            assert_grad_parity(mine[i], r32[i], r64[i], "d/d" + name, tol=2e-5, case=case)
        else:
            assert mine[i] is None
    if n * c * h * w <= 300:
        model = np.stack([PM.ssim_map(x0[b].double().numpy(), y0[b].double().numpy()) for b in range(n)])
        check_pixel_model(mine[0], r32[0], model, case, "ssim")


SMOOTH_SHAPES = [(1, 2, 2), (2, 15, 119), (2, 16, 120), (2, 17, 121), (3, 33, 241), (12, 192, 640)]


@pytest.mark.parametrize("img_grad", [False, True], ids=["img_const", "img_grad"])
@pytest.mark.parametrize("shape", SMOOTH_SHAPES, ids=["x".join(map(str, s)) for s in SMOOTH_SHAPES])
def test_smooth_loss_sweep(shape, img_grad, cuda_device):
    dev = cuda_device
    B, H, W = shape
    case = f"smooth/{B}x{H}x{W}/{'img_grad' if img_grad else 'img_const'}"
    gen = torch.Generator().manual_seed(B * H * W)
    d0 = 0.05 + torch.rand(B, 1, H, W, generator=gen)
    i0 = torch.rand(B, 3, H, W, generator=gen)
    i0[..., W // 2] = i0[..., W // 2 - 1]          # a column without an image edge

    def run(d, img, fn):
        d, img = _leaf(d), img.detach().clone().requires_grad_(img_grad)
        loss = fn(d, img)
        (2.5 * loss).backward()
        return loss.detach(), d.grad, img.grad

    mine = run(d0.to(dev), i0.to(dev), L.get_smooth_loss)
    _sync(dev)
    r32 = run(d0, i0, O.smooth_loss)
    r64 = run(d0.double(), i0.double(), O.smooth_loss)
    check_forward(mine[0].reshape(1), r32[0].reshape(1), r64[0].reshape(1), case, "loss")
    assert_grad_parity(mine[1], r32[1], r64[1], "d/d disp", case=case)
    if img_grad:
        assert_grad_parity(mine[2], r32[2], r64[2], "d/d img", case=case)
    else:
        assert mine[2] is None


def _aten_grid_sample(img, grid):
    return F.grid_sample(img, grid, align_corners=True, padding_mode="border")


GS_CASES = {
    "runs_2x3x10x14_to_96x160": ((2, 3, 10, 14), (96, 160)),     # many outputs per source pixel
    "frame_4x3x192x640_to_48x80": ((4, 3, 192, 640), (48, 80)),
    "past_cap_3x3x96x320_to_320x640": ((3, 3, 96, 320), (320, 640)),   # n*Ho*Wo = 614,400 > 606,208
    "edge_1x2x5x4_to_12x11": ((1, 2, 5, 4), (12, 11)),          # pixel-model size
}


def _gs_grid(n, ho, wo, gen):
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, ho), torch.linspace(-1, 1, wo), indexing="ij")
    base = torch.stack([xs, ys], -1).unsqueeze(0).repeat(n, 1, 1, 1) * 1.05
    base = base + 0.03 * torch.randn(n, ho, wo, 2, generator=gen)
    base[:, 0, :, 1], base[:, :, 0, 0] = -1.0, -1.0                     # exactly on the border
    base[:, -1, :, 1], base[:, :, -1, 0] = 1.0, 1.0
    base[:, ho // 2, : wo // 3] = torch.tensor([-3.0, 2.5])            # far outside: clamped onto border pixels
    base[:, ho // 3, wo // 2:] = torch.tensor([1.0 + 1e-7, -1.0 - 1e-7])
    return base


@pytest.mark.parametrize("name", list(GS_CASES))
def test_grid_sample_sweep(name, cuda_device):
    dev = cuda_device
    (n, c, h, w), (ho, wo) = GS_CASES[name]
    case = "grid_sample/" + name
    gen = torch.Generator().manual_seed(len(name))
    img0 = torch.rand(n, c, h, w, generator=gen)
    base = _gs_grid(n, ho, wo, gen)
    up = torch.rand(n, c, ho, wo, generator=gen) - 0.3
    if n * ho * wo > GRID_CAP_THREADS:
        assert name.startswith("past_cap")

    def run(img, grid, fn):
        img, raw = _leaf(img), _leaf(grid.permute(0, 3, 1, 2).contiguous())   # Project3D's (n,H,W,2) view of (n,2,H,W)
        out = fn(img, raw.permute(0, 2, 3, 1))
        (out * up.to(out.device, out.dtype)).sum().backward()
        return out.detach(), raw.grad.permute(0, 2, 3, 1), img.grad

    mine = run(img0.to(dev), base.to(dev), L.grid_sample)
    _sync(dev)
    r32 = run(img0, base, _aten_grid_sample)
    r64 = run(img0.double(), base.double(), _aten_grid_sample)
    check_forward(mine[0], r32[0], r64[0], case, "out")
    assert_grad_parity(mine[1], r32[1], r64[1], "d/d grid", case=case)
    assert_grad_parity(mine[2], r32[2], r64[2], "d/d images", case=case)
    if n * c * ho * wo <= 300:
        model = [PM.grid_sample_border(img0[b].double().numpy(), base[b].double().numpy(), up[b].double().numpy())
                 for b in range(n)]
        check_pixel_model(mine[0], r32[0], np.stack([m[0] for m in model]), case, "out")
        check_pixel_model(mine[1], r32[1], np.stack([m[1] for m in model]), case, "d/d grid", grad=True)


@pytest.mark.parametrize("invert", [False, True], ids=["T", "T_inv"])
@pytest.mark.parametrize("n", [1, 64, 65, 1000])
def test_transformation_from_parameters_sweep(n, invert, cuda_device):
    dev = cuda_device
    case = f"pose/n{n}/{'invert' if invert else 'forward'}"
    gen = torch.Generator().manual_seed(n + invert)
    aa0, tr0 = 0.3 * torch.randn(n, 1, 3, generator=gen), torch.randn(n, 1, 3, generator=gen)
    zero = (torch.arange(n) % 7) == 1                        # zero rotation: a legal network output
    aa0[zero] = 0.0
    up = torch.randn(n, 4, 4, generator=gen)

    def run(aa, tr, fn):
        aa, tr = _leaf(aa), _leaf(tr)
        T = fn(aa, tr, invert)
        (T * up.to(T.device, T.dtype)).sum().backward()
        return T.detach(), aa.grad, tr.grad

    mine = run(aa0.to(dev), tr0.to(dev), L.transformation_from_parameters)
    _sync(dev)
    r32 = run(aa0, tr0, O.transformation_from_parameters)
    r64 = run(aa0.double(), tr0.double(), O.transformation_from_parameters)
    check_forward(mine[0], r32[0], r64[0], case, "T")
    # at angle 0 the reference's gradient w.r.t. the axis-angle is that of its 1e-7-regularised division, not
    # the rotation's derivative: those rows are only required to be finite
    keep = ~zero
    if bool(keep.any()):
        k = keep.to(mine[1].device)
        assert_grad_parity(mine[1][k], r32[1][keep], r64[1][keep], "d/d axisangle", case=case)
    assert bool(torch.isfinite(mine[1]).all())
    assert_grad_parity(mine[2], r32[2], r64[2], "d/d translation", case=case)


# ------------------------------------------------------------------------------------------------------------------
# c. determinism and streams
# ------------------------------------------------------------------------------------------------------------------
def _det_inputs(name, gen):
    if name == "backproject_project":
        n, H, W = 4, 192, 640
        K, inv_K = _camera(n, H, W, gen)
        return dict(depth=1 + 5 * torch.rand(n, 1, H, W, generator=gen), K=K, inv_K=inv_K,
                    aa=0.05 * torch.randn(n, 1, 3, generator=gen), tr=0.1 * torch.randn(n, 1, 3, generator=gen),
                    up=torch.rand(n, H, W, 2, generator=gen))
    if name == "ssim":
        s = (4, 3, 192, 640)
        return dict(x=torch.rand(*s, generator=gen), y=torch.rand(*s, generator=gen), up=torch.rand(*s, generator=gen))
    if name == "smooth":
        return dict(disp=0.05 + torch.rand(12, 1, 192, 640, generator=gen), img=torch.rand(12, 3, 192, 640, generator=gen))
    if name == "grid_sample":
        return dict(img=torch.rand(4, 3, 192, 640, generator=gen), grid=_gs_grid(4, 192, 640, gen),
                    up=torch.rand(4, 3, 192, 640, generator=gen))
    if name == "pose":
        return dict(aa=0.3 * torch.randn(1000, 1, 3, generator=gen), tr=torch.randn(1000, 1, 3, generator=gen),
                    up=torch.randn(1000, 4, 4, generator=gen))
    raise KeyError(name)


def _det_run(name, x):
    """Forward + backward of one tier-A operator on device inputs `x`; every output and gradient."""
    if name == "backproject_project":
        d, a, t = (x[k].detach().requires_grad_(True) for k in ("depth", "aa", "tr"))
        n, _, H, W = d.shape
        T = L.transformation_from_parameters(a, t)
        grid = L.Project3D(n, H, W)(L.BackprojectDepth(n, H, W)(d, x["inv_K"]), x["K"], T)
        (grid * x["up"]).sum().backward()
        return [grid, d.grad, a.grad, t.grad]
    if name == "ssim":
        a, b = x["x"].detach().requires_grad_(True), x["y"].detach().requires_grad_(True)
        out = L.SSIM()(a, b)
        (out * x["up"]).sum().backward()
        return [out, a.grad, b.grad]
    if name == "smooth":
        d, img = x["disp"].detach().requires_grad_(True), x["img"].detach().requires_grad_(True)
        loss = L.get_smooth_loss(d, img)
        loss.backward()
        return [loss, d.grad, img.grad]
    if name == "grid_sample":
        img, raw = x["img"].detach().requires_grad_(True), x["grid"].permute(0, 3, 1, 2).detach().requires_grad_(True)
        out = L.grid_sample(img, raw.permute(0, 2, 3, 1))
        (out * x["up"]).sum().backward()
        return [out, img.grad, raw.grad]
    a, t = x["aa"].detach().requires_grad_(True), x["tr"].detach().requires_grad_(True)
    T = L.transformation_from_parameters(a, t, True)
    (T * x["up"]).sum().backward()
    return [T, a.grad, t.grad]


@pytest.mark.parametrize("name", ["backproject_project", "ssim", "smooth", "grid_sample", "pose"])
def test_backward_bit_identical_and_on_the_callers_stream(name, cuda_device):
    """Two runs on the default stream give the same bits; so does a run on a side stream whose inputs are written
    by a copy queued behind ~0.1 s of GPU sleep on that stream.  A kernel enqueued on another stream than the
    caller's would read the NaN the input buffers held before the copy."""
    dev = cuda_device
    base = {k: v.to(dev) for k, v in _det_inputs(name, torch.Generator().manual_seed(17)).items()}
    torch.cuda.synchronize()
    first = [t.detach().clone() for t in _det_run(name, base)]
    second = [t.detach().clone() for t in _det_run(name, base)]
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(first, second)):
        assert torch.equal(a, b), (name, i)
    side = torch.cuda.Stream()
    staged = {k: torch.full_like(v, float("nan")) for k, v in base.items()}
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        for k, v in staged.items():
            v.record_stream(side)
            v.copy_(base[k])
        on_side = [t.detach().clone() for t in _det_run(name, staged)]
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(first, on_side)):
        assert torch.equal(a, b), (name, "side stream", i)


# ------------------------------------------------------------------------------------------------------------------
# d. bbd_smooth_fused in tier B's form
# ------------------------------------------------------------------------------------------------------------------
def _pyramid(B, H, W, gen):
    disps = [0.02 + torch.rand(B, 1, H >> s, W >> s, generator=gen) for s in range(4)]
    imgs = [torch.rand(B, 3, H >> s, W >> s, generator=gen) for s in range(4)]
    return disps, imgs


def smooth_fused_direct(be, disps, imgs, defer_norm):
    """bbd_smooth_fused over all levels at once with normalize=1, as the fused loss calls it; with defer_norm the
    gradient is finished here, g * coef[0] - coef[1], as the disparity backward finishes it there."""
    S, B = len(disps), disps[0].shape[0]
    dev = disps[0].device
    sa = _lib.SmoothArgs()
    sa.batch, sa.levels, sa.normalize = B, S, 1
    gdisp = [torch.empty_like(d) for d in disps]
    for l in range(S):
        sa.h[l], sa.w[l] = disps[l].shape[2], disps[l].shape[3]
        sa.disp[l], sa.img[l], sa.gdisp[l] = disps[l].data_ptr(), imgs[l].data_ptr(), gdisp[l].data_ptr()
    hs, ws = (C.c_int32 * S)(*[d.shape[2] for d in disps]), (C.c_int32 * S)(*[d.shape[3] for d in disps])
    scratch = torch.empty(max(1, be.value("smooth_scratch_floats", B, S, hs, ws)), device=dev)
    loss = torch.empty(S, device=dev)
    sa.scratch, sa.loss = scratch.data_ptr(), loss.data_ptr()
    coef = None
    if defer_norm:
        coef = torch.empty(S, B, 2, device=dev)
        sa.defer_norm, sa.coef = 1, coef.data_ptr()
    be.call("smooth_fused", C.byref(sa))
    if defer_norm:
        gdisp = [g * coef[l, :, 0].view(B, 1, 1, 1) - coef[l, :, 1].view(B, 1, 1, 1) for l, g in enumerate(gdisp)]
    return loss, gdisp


def smooth_reference(disps, imgs, dtype, chunk=16):
    """Per level: O.smooth_loss(disp / (mean_hw(disp) + 1e-7), img) (trainer.py:560-563) and its gradient w.r.t.
    disp, evaluated over chunks of samples (the loss is a mean over equally sized samples)."""
    losses, grads = [], []
    for d_all, i_all in zip(disps, imgs):
        B = d_all.shape[0]
        tot, gs = 0.0, []
        for b0 in range(0, B, chunk):
            d = _leaf(d_all[b0:b0 + chunk], dtype=dtype)
            img = i_all[b0:b0 + chunk].to(dtype)
            norm = d / (d.mean(2, True).mean(3, True) + 1e-7)
            part = O.smooth_loss(norm, img) * (d.shape[0] / B)
            part.backward()
            tot += float(part.detach())
            gs.append(d.grad)
        losses.append(tot)
        grads.append(torch.cat(gs))
    return losses, grads


_SMOOTH_REF = {}


@pytest.mark.parametrize("batch", [1, 12, 256])
@pytest.mark.parametrize("frame", [(64, 96), (192, 640)], ids=["64x96", "192x640"])
def test_smooth_fused_levels_tier_b_form(frame, batch, cuda_device):
    dev = cuda_device
    H, W = frame
    disps, imgs = _pyramid(batch, H, W, torch.Generator().manual_seed(batch + H))
    r32 = smooth_reference(disps, imgs, torch.float32)
    r64 = smooth_reference(disps, imgs, torch.float64)
    be = L._backend()
    dd, di = [d.to(dev) for d in disps], [i.to(dev) for i in imgs]
    for defer in (0, 1):
        case = f"smooth_fused/{H}x{W}/b{batch}/defer{defer}"
        loss, gdisp = smooth_fused_direct(be, dd, di, defer)
        _sync(dev)
        for l in range(4):
            got, want = float(loss[l]), r64[0][l]
            ok = abs(got - want) <= 2e-6 * max(1.0, abs(want))
            PARITY_LOG.append({"case": case, "key": f"loss level {l}", "loss": got, "f64": want, "fp32_aten": r32[0][l],
                               "bar": "rel<=2e-6 vs f64", "passed": ok})
            assert ok, (case, l, got, want, r32[0][l])
            assert_grad_parity(gdisp[l], r32[1][l], r64[1][l], f"d/d disp level {l}", case=case)


# ------------------------------------------------------------------------------------------------------------------
# e. bbd_u8_to_f32 on the device
# ------------------------------------------------------------------------------------------------------------------
# 16 * 606,208 + 7: exactly one full pass of the 16-byte kernel plus a 7-byte tail; 16 * (2 * 606,208 + 3) + 9:
# a second grid-stride pass
U8_LENGTHS = [1, 15, 16, 17, 33, 65541, 16 * 606208 + 7, 16 * (2 * 606208 + 3) + 9]


@pytest.mark.parametrize("n", U8_LENGTHS)
def test_u8_to_f32_offsets_and_lengths(n, cuda_device):
    """Every source offset 0..15 bytes and destination offset 0/4/8/12 bytes: bit-identical to x.float().div(255),
    and nothing written outside [dst, dst + n)."""
    dev = cuda_device
    be = L._backend()
    gen = torch.Generator().manual_seed(n % 9973)
    host = torch.randint(0, 256, (n + 16,), generator=gen, dtype=torch.uint8)
    host[: min(256, n + 16)] = torch.arange(min(256, n + 16), dtype=torch.uint8)   # every code at least once
    want = host.float().div(255).to(dev)
    src = host.to(dev)
    dst = torch.empty(n + 8, device=dev)
    for so in range(16):
        for do in range(4):
            dst.fill_(float("nan"))
            be.call("u8_to_f32", C.c_void_p(src.data_ptr() + so), C.c_void_p(dst.data_ptr() + 4 * do), C.c_size_t(n))
            assert torch.equal(dst[do:do + n], want[so:so + n]), (n, so, do)
            assert bool(dst[:do].isnan().all()) and bool(dst[do + n:].isnan().all()), (n, so, do)
