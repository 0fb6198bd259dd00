"""Parity of the sm_100a kernels (through the C ABI) against the oracle -- runs on the B200 box.

Bars (BASELINE.md 5): loss within 1e-5 relative (we hold 2e-6); gradients within 1e-5
relative L2 against the fp32 oracle; argmin selections identical wherever the oracle's
margin between its two best candidates exceeds 1e-6.
"""
import pytest
import torch

from baseboostdepth_b200.synthetic import make_batch, make_noise
from baseboostdepth_b200.trainer import materialise_warps, plan_for
from fused_util import mirror_to_device, retain_pose_grads, run_fused, to_device
from helpers import (PARITY_LOG, Golden, assert_grad_parity, golden_cases, max_abs, near_tie_mask, pixel_agreement, rel_l2,
                     selection_check)
from oracle import loss_path as O

pytestmark = pytest.mark.gpu
CASES = golden_cases()


@pytest.mark.parametrize("case", CASES)
def test_golden_case_on_gpu(case, cuda_device):
    g = Golden(case)
    retain_pose_grads(g.outputs)
    ref, aux = O.run(g.inputs, g.outputs, g.opt(), g.noise, num_scales=g.num_scales)
    ref["loss"].backward()
    g64 = Golden(case, dtype=torch.float64)
    retain_pose_grads(g64.outputs)
    ref64, _ = O.run(g64.inputs, g64.outputs, g64.opt(), g64.noise, num_scales=g.num_scales)
    ref64["loss"].backward()

    h = Golden(case)
    hi, ho, leaves = mirror_to_device(h.inputs, h.outputs, h.params, cuda_device)
    noise = {k: v.to(cuda_device) for k, v in h.noise.items()}
    losses, plan = run_fused(hi, ho, h.opt(), noise, h.num_scales, groups=aux["groups"])
    for k, v in g.losses.items():
        assert abs(float(losses[k]) - v) <= 2e-6 * max(1.0, abs(v)), (k, float(losses[k]), v)
    losses["loss"].backward()
    torch.cuda.synchronize()
    for k, leaf in leaves.items():
        ref32 = g.params[k].grad if k[0] == "disp" else g.outputs[k].grad
        ref64_ = g64.params[k].grad if k[0] == "disp" else g64.outputs[k].grad
        assert_grad_parity(leaf.grad, ref32, ref64_, k, case=case)
    selection_check(ho["argmin"], plan, aux, h.scales)
    h.inputs, h.outputs = hi, ho
    with torch.no_grad():
        materialise_warps(h.inputs, h.outputs, h.opt(), plan)
    s0 = h.scales[0]
    for f in plan.frames:
        assert max_abs(h.outputs[("color", f, s0)], g.ref_out[("color", f, s0)]) <= 2e-5, f


def test_far_baselines_that_never_win_on_gpu(cuda_device):
    """Tri-min batch at frame size whose +-2 / +-3 frames are far from the target: their candidate pairs win nowhere,
    the many-candidate kernel skips their sweeps of the gradient round.  Loss, selections and gradients against the
    oracle on the same inputs; the poses of the skipped candidates get exactly zero gradient."""
    cfg = dict(batch=4, height=192, width=640, baselines=[3, 2, 1, 3], trimin=True, decomp=False)
    scales = [0, 1, 2, 3]
    opt = O.default_opt(height=192, width=640, trimin=True, decomp=False, pose_error=5.5, scales=scales, batch_size=4)

    def build():
        inputs, outputs, params = make_batch(seed=21, device="cpu", scales=scales, **cfg)
        for k in list(inputs):
            if isinstance(k, tuple) and k[0] == "color" and k[1] in (2, -2, 3, -3):
                inputs[k] = inputs[k] + 3.0
        return inputs, outputs, params
    inputs, outputs, params = build()
    plan = plan_for(inputs["ordering"], True, False, None)
    noise = make_noise(plan, 192, 640, seed=22)
    retain_pose_grads(outputs)
    ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()
    i64, o64, p64 = make_batch(seed=21, device="cpu", dtype=torch.float64, scales=scales, **cfg)
    for k in list(i64):
        if isinstance(k, tuple) and k[0] == "color" and k[1] in (2, -2, 3, -3):
            i64[k] = i64[k] + 3.0
    retain_pose_grads(o64)
    ref64, _ = O.run(i64, o64, opt, {k: v.double() for k, v in noise.items()}, num_scales=4)
    ref64["loss"].backward()
    gi, go, leaves = mirror_to_device(inputs, outputs, params, cuda_device)
    losses, plan = run_fused(gi, go, opt, {k: v.to(cuda_device) for k, v in noise.items()}, 4, groups=aux["groups"])
    losses["loss"].backward()
    torch.cuda.synchronize()
    for k in ref:
        assert abs(float(losses[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), k
    selection_check(go["argmin"], plan, aux, scales)
    zero_poses = 0
    for k, leaf in leaves.items():
        want = params[k].grad if k[0] == "disp" else outputs[k].grad
        if float(want.abs().max()) == 0.0:
            assert float(leaf.grad.abs().max()) == 0.0, k
            zero_poses += 1
        else:
            r64 = p64[k].grad if k[0] == "disp" else o64[k].grad
            assert_grad_parity(leaf.grad, want, r64, k, case="far_baselines_640x192_b4")
    assert zero_poses > 0   # the far frames' poses: nothing was warped with them successfully


FULL = [
    ("config2_640x192_b4", dict(batch=4, height=192, width=640, baselines=[1] * 4, trimin=False, decomp=False)),
    ("config3a_trimin_mixed_b4", dict(batch=4, height=192, width=640, baselines=[3, 2, 1, "s"], trimin=True,
                                      decomp=False)),
    ("config3b_decomp_b3", dict(batch=3, height=192, width=640, baselines=[3, 2, "s"], trimin=True, decomp=True)),
    ("config4_1024x320_b1", dict(batch=1, height=320, width=1024, baselines=[1], trimin=False, decomp=False)),
    ("ragged_200x330_b2", dict(batch=2, height=200, width=330, baselines=[1, 2], trimin=True, decomp=False,
                               scales=(0,))),
]


@pytest.mark.parametrize("name,cfg", FULL, ids=[n for n, _ in FULL])
def test_full_size_against_oracle(name, cfg, cuda_device):
    cfg = dict(cfg)
    scales = list(cfg.pop("scales", (0, 1, 2, 3)))
    opt = O.default_opt(height=cfg["height"], width=cfg["width"], trimin=cfg["trimin"], decomp=cfg["decomp"],
                        pose_error=5.5, scales=scales, batch_size=cfg["batch"])
    inputs, outputs, params = make_batch(seed=21, device="cpu", scales=scales, **cfg)
    plan = plan_for(inputs["ordering"], opt.trimin, opt.decomp,
                    inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
    noise = make_noise(plan, cfg["height"], cfg["width"], seed=5)
    retain_pose_grads(outputs)
    ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()
    i64, o64, p64 = make_batch(seed=21, device="cpu", dtype=torch.float64, scales=scales, **cfg)
    retain_pose_grads(o64)
    ref64, _ = O.run(i64, o64, opt, {k: v.double() for k, v in noise.items()}, num_scales=4)
    ref64["loss"].backward()

    gi, go, leaves = mirror_to_device(inputs, outputs, params, cuda_device)
    gnoise = {k: v.to(cuda_device) for k, v in noise.items()}
    losses, plan = run_fused(gi, go, opt, gnoise, 4, groups=aux["groups"])
    losses["loss"].backward()
    torch.cuda.synchronize()
    for k in ref:
        assert abs(float(losses[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), k
    for k, leaf in leaves.items():
        ref32 = params[k].grad if k[0] == "disp" else outputs[k].grad
        r64 = p64[k].grad if k[0] == "disp" else o64[k].grad
        assert_grad_parity(leaf.grad, ref32, r64, k, case=name)
        if k[0] == "disp":   # per-pixel: all but the footprints of a few near-ties agree to 1e-4 of the peak
            frac = pixel_agreement(leaf.grad, ref32, tol=1e-4)
            assert frac <= 5e-3 * (1 + k[1]), (k, frac)
    selection_check(go["argmin"], plan, aux, scales)


# ---- the benchmarked workloads at full size (BASELINE.json configs 2-4, synthetic.WORKLOADS) ----------------
from baseboostdepth_b200.synthetic import WORKLOADS  # noqa: E402


@pytest.mark.parametrize("name", list(WORKLOADS))
def test_benched_workload_against_oracle(name, cuda_device):
    """The exact batch bench.py times (same WORKLOADS entry, full batch, all scales) against the oracle:
    loss 2e-6, argmin identical wherever the oracle's margin exceeds 1e-6, gradients to the logged bar,
    and per pixel at scale 0: outside the 1-dilated set of near-ties the disparity gradient agrees to 1e-5 of
    its peak for all but a vanishing fraction of pixels (reported in the parity log)."""
    batch, H, W, baselines, trimin, decomp = WORKLOADS[name]
    scales = [0, 1, 2, 3]
    opt = O.default_opt(height=H, width=W, trimin=trimin, decomp=decomp, pose_error=5.5, scales=scales, batch_size=batch)
    cfg = dict(batch=batch, height=H, width=W, baselines=list(baselines), trimin=trimin, decomp=decomp)
    inputs, outputs, params = make_batch(seed=1234, device="cpu", scales=scales, **cfg)
    plan = plan_for(inputs["ordering"], opt.trimin, opt.decomp,
                    inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
    noise = make_noise(plan, H, W, seed=4321)
    retain_pose_grads(outputs)
    ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()
    i64, o64, p64 = make_batch(seed=1234, device="cpu", dtype=torch.float64, scales=scales, **cfg)
    retain_pose_grads(o64)
    ref64, _ = O.run(i64, o64, opt, {k: v.double() for k, v in noise.items()}, num_scales=4)
    ref64["loss"].backward()

    gi, go, leaves = mirror_to_device(inputs, outputs, params, cuda_device)
    gnoise = {k: v.to(cuda_device) for k, v in noise.items()}
    losses, plan = run_fused(gi, go, opt, gnoise, 4, groups=aux["groups"])
    losses["loss"].backward()
    torch.cuda.synchronize()
    for k in ref:
        assert abs(float(losses[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), (k, float(losses[k]), float(ref[k]))
    for k, leaf in leaves.items():
        ref32 = params[k].grad if k[0] == "disp" else outputs[k].grad
        r64 = p64[k].grad if k[0] == "disp" else o64[k].grad
        assert_grad_parity(leaf.grad, ref32, r64, k, case=name)
    selection_check(go["argmin"], plan, aux, scales)
    # per-pixel bar at full resolution
    near = near_tie_mask(plan, aux, 0)
    g_mine, g_ref = leaves[("disp", 0)].grad.cpu()[:, 0].double(), params[("disp", 0)].grad[:, 0].double()
    off = (g_mine - g_ref).abs() > 1e-5 * g_ref.abs().max()
    frac_near = near.double().mean().item()
    frac_off_outside = (off & ~near).double().mean().item()
    PARITY_LOG.append({"case": name, "key": "per-pixel d loss/d disp_0", "near_tie_fraction_dilated": frac_near,
                       "pixels_off_by_1e-5_of_peak_outside_near_ties": frac_off_outside,
                       "pixels_off_anywhere": off.double().mean().item()})
    assert frac_near < 2e-3, frac_near
    assert frac_off_outside <= 1e-4, frac_off_outside


def test_pipelined_form_on_gpu(cuda_device, monkeypatch):
    """The opt-in three-warp form of the fused kernel (BBD_PIPE=1, csrc/bbd_pipe.cuh) at the benchmark size: loss and
    gradients against the one-warp streaming form of the same launch (same arithmetic up to the reciprocal's
    range handling, same order of adding) and against the oracle."""
    batch, H, W, baselines, trimin, decomp = WORKLOADS["kitti_640x192_b12_pm1"]
    scales = [0, 1, 2, 3]
    opt = O.default_opt(height=H, width=W, trimin=trimin, decomp=decomp, pose_error=5.5, scales=scales, batch_size=batch)
    cfg = dict(batch=batch, height=H, width=W, baselines=list(baselines), trimin=trimin, decomp=decomp)
    inputs, outputs, params = make_batch(seed=77, device="cpu", scales=scales, **cfg)
    plan = plan_for(inputs["ordering"], opt.trimin, opt.decomp, None)
    noise = make_noise(plan, H, W, seed=78)
    retain_pose_grads(outputs)
    ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()
    gnoise = {k: v.to(cuda_device) for k, v in noise.items()}
    got = {}
    for form in ("1", "0"):
        monkeypatch.setenv("BBD_PIPE", form)
        gi, go, leaves = mirror_to_device(inputs, outputs, params, cuda_device)
        losses, _ = run_fused(gi, go, opt, gnoise, 4, groups=aux["groups"])
        losses["loss"].backward()
        torch.cuda.synchronize()
        got[form] = (losses, leaves, go["argmin"].clone())
    lp, gp, wp = got["1"]
    ls, gs, ws = got["0"]
    for k in ref:
        assert abs(float(lp[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), k
        assert abs(float(lp[k]) - float(ls[k])) <= 2e-7 * max(1.0, abs(float(ls[k]))), k
    for k in gp:
        assert rel_l2(gp[k].grad, gs[k].grad) <= 2e-6, (k, rel_l2(gp[k].grad, gs[k].grad))
    assert (wp != ws).float().mean().item() <= 1e-5


def test_projected_coordinates_bit_exact(cuda_device):
    """north_star clause 1: projected pixel coordinates / tap indices are bit-identical to the reference's.
    Both projection chains of the library -- the tile kernels' (bbd_warp_forward) and the streaming kernel's
    (bbd_project_coords) -- against Project3D's grid (layers.py:181-195) and ATen's unnormalise + clip + floor
    (F.grid_sample, trainer.py:442), at the benchmark size, scales 0 and 3, frames +-1."""
    import ctypes as C
    from baseboostdepth_b200 import _lib
    be = _lib.cuda_backend()
    batch, H, W, baselines, trimin, decomp = WORKLOADS["kitti_640x192_b12_pm1"]
    opt = O.default_opt(height=H, width=W, batch_size=batch)
    inputs, outputs, params = make_batch(seed=77, device="cpu", batch=batch, height=H, width=W, baselines=list(baselines))
    ref_out = dict(outputs)
    with torch.no_grad():
        ordering = inputs["ordering"]
        masks = O.sub_batch_masks(ordering, O.frame_ids_from_ordering(ordering), O.initial_valid_frames(ordering), opt.trimin)
        O.view_synthesis(inputs, ref_out, opt, masks)
    dev = cuda_device
    K, inv_K = inputs[("K", 0)].to(dev), inputs[("inv_K", 0)].to(dev).contiguous()
    for s in (0, 3):
        depth = ref_out[("depth", 0, s)].to(dev).contiguous()
        for f in (1, -1):
            T = outputs[("cam_T_cam", 0, f)].detach()
            P = torch.matmul(inputs[("K", 0)], T)[:, :3, :].contiguous().to(dev)
            want = ref_out[("grid", f, s)]                                    # (n,H,W,2)
            ix = ((want[..., 0] + 1) / 2 * (W - 1)).clamp(0, W - 1)
            iy = ((want[..., 1] + 1) / 2 * (H - 1)).clamp(0, H - 1)
            grid = torch.empty(batch, 2, H, W, device=dev)
            pix = torch.empty(batch, 2, H, W, device=dev)
            be.call("project_coords", batch, H, W, C.c_void_p(depth.data_ptr()), C.c_void_p(inv_K.data_ptr()),
                    C.c_void_p(P.data_ptr()), C.c_void_p(grid.data_ptr()), C.c_void_p(pix.data_ptr()))
            warped = torch.empty(batch, 3, H, W, device=dev)
            grid2 = torch.empty(batch, 2, H, W, device=dev)
            src = inputs[("color", f, 0)].to(dev).contiguous()
            be.call("warp_forward", batch, H, W, C.c_void_p(src.data_ptr()), C.c_void_p(depth.data_ptr()),
                    C.c_void_p(inv_K.data_ptr()), C.c_void_p(P.data_ptr()), C.c_void_p(warped.data_ptr()),
                    C.c_void_p(grid2.data_ptr()))
            torch.cuda.synchronize()
            for g in (grid, grid2):
                assert torch.equal(g.cpu().permute(0, 2, 3, 1), want), (s, f)
            assert torch.equal(pix[:, 0].cpu(), ix) and torch.equal(pix[:, 1].cpu(), iy), (s, f)
            assert torch.equal(pix[:, 0].cpu().floor(), ix.floor()) and torch.equal(pix[:, 1].cpu().floor(), iy.floor())


def test_deterministic_and_linear(cuda_device):
    """Size-independent properties at the benchmark size: bit-identical reruns (no float atomics)
    and gradients linear in the upstream gradient."""
    cfg = dict(batch=12, height=192, width=640, baselines=[1] * 12, trimin=False, decomp=False)
    opt = O.default_opt()
    runs = []
    for scale in (1.0, 1.0, 3.0):
        gi, go, gp = make_batch(seed=3, device=cuda_device, **cfg)
        plan = plan_for(gi["ordering"], False, False, None)
        noise = {k: v.to(cuda_device) for k, v in make_noise(plan, 192, 640, seed=8).items()}
        losses, _ = run_fused(gi, go, opt, noise, 4)
        (losses["loss"] * scale).backward()
        torch.cuda.synchronize()
        runs.append((float(losses["loss"]), {k: v.grad.clone() for k, v in gp.items()}))
    assert runs[0][0] == runs[1][0]
    for k in runs[0][1]:
        assert torch.equal(runs[0][1][k], runs[1][1][k]), k
        assert rel_l2(runs[2][1][k], 3.0 * runs[0][1][k]) <= 1e-6, k


def test_sample_independence(cuda_device):
    """Each sample is an independent unit (SURVEY 8e): the loss of a batch is the mean of the losses
    of its halves -- the property the batch sharding across GPUs relies on."""
    cfg = dict(height=96, width=320, trimin=False, decomp=False)
    opt = O.default_opt(height=96, width=320)
    gi, go, gp = make_batch(seed=4, device=cuda_device, batch=4, baselines=[1] * 4, **cfg)
    plan = plan_for(gi["ordering"], False, False, None)
    noise = {k: v.to(cuda_device) for k, v in make_noise(plan, 96, 320, seed=9).items()}
    with torch.no_grad():
        full, _ = run_fused(gi, go, opt, noise, 4)
        halves = []
        for lo in (0, 2):
            hi_ = {k: (v[lo:lo + 2] if torch.is_tensor(v) and v.shape[0] == 4 else v) for k, v in gi.items()}
            hi_["ordering"] = gi["ordering"][lo:lo + 2]
            ho = {k: (v[lo:lo + 2] if torch.is_tensor(v) and v.shape[0] == 4 else v) for k, v in go.items()}
            hn = {k: v[lo:lo + 2] for k, v in noise.items()}
            part, _ = run_fused(hi_, ho, opt, hn, 4)
            halves.append(float(part["loss"]))
    assert abs(float(full["loss"]) - 0.5 * (halves[0] + halves[1])) <= 1e-6


def test_cuda_required():
    from baseboostdepth_b200 import _lib
    be = _lib.cuda_backend()
    with pytest.raises(RuntimeError):
        be.check_device(torch.zeros(1))


@pytest.mark.parametrize("invert", [False, True])
def test_pose_kernel_on_gpu(invert, cuda_device):
    import baseboostdepth_b200.layers as L
    from baseboostdepth_b200 import geometry as G
    gen = torch.Generator().manual_seed(3)
    aa0, tr0 = 0.2 * torch.randn(24, 1, 3, generator=gen), torch.randn(24, 1, 3, generator=gen)
    w = torch.randn(24, 4, 4, generator=gen)
    aa_c, tr_c = aa0.clone().requires_grad_(True), tr0.clone().requires_grad_(True)
    Tc = G.transformation_from_parameters(aa_c, tr_c, invert)
    (Tc * w).sum().backward()
    aa_g, tr_g = aa0.to(cuda_device).requires_grad_(True), tr0.to(cuda_device).requires_grad_(True)
    Tg = L.transformation_from_parameters(aa_g, tr_g, invert)
    (Tg * w.to(cuda_device)).sum().backward()
    assert max_abs(Tg, Tc) <= 5e-7
    assert rel_l2(aa_g.grad, aa_c.grad) <= 1e-5 and rel_l2(tr_g.grad, tr_c.grad) <= 1e-5


def test_tier_a_operators_on_gpu(cuda_device):
    """Module-level drop-ins (layers.py names) against the oracle's ATen ops, on the device."""
    import baseboostdepth_b200.layers as L
    gen = torch.Generator().manual_seed(5)
    n, H, W = 3, 48, 96
    K = torch.tensor([[0.58 * W, 0, 0.5 * W, 0], [0, 1.92 * H, 0.5 * H, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]]).repeat(n, 1, 1)
    inv_K = torch.linalg.pinv(K)
    from baseboostdepth_b200 import geometry as G
    Tm = G.transformation_from_parameters(0.02 * torch.randn(n, 1, 3, generator=gen), 0.05 * torch.randn(n, 1, 3, generator=gen))
    depth = 1 + 5 * torch.rand(n, 1, H, W, generator=gen)
    x, y = torch.rand(n, 3, H, W, generator=gen), torch.rand(n, 3, H, W, generator=gen)
    # oracle on CPU
    d_c = depth.clone().requires_grad_(True)
    pix_c = O.project(O.backproject(d_c, inv_K, H, W), K, Tm, H, W)
    x_c = x.clone().requires_grad_(True)
    s_c = O.ssim(x_c, y)
    (pix_c.sum() + s_c.sum()).backward()
    # kernels on GPU
    dev = cuda_device
    d_g = depth.to(dev).requires_grad_(True)
    pix_g = L.Project3D(n, H, W)(L.BackprojectDepth(n, H, W)(d_g, inv_K.to(dev)), K.to(dev), Tm.to(dev))
    x_g = x.to(dev).requires_grad_(True)
    s_g = L.SSIM()(x_g, y.to(dev))
    (pix_g.sum() + s_g.sum()).backward()
    assert max_abs(pix_g, pix_c) <= 1e-6 and max_abs(s_g, s_c) <= 1e-6
    assert rel_l2(d_g.grad, d_c.grad) <= 1e-5 and rel_l2(x_g.grad, x_c.grad) <= 2e-5
    norm = torch.rand(n, 1, H, W, generator=gen)
    assert abs(float(L.get_smooth_loss(norm.to(dev), x.to(dev))) - float(O.smooth_loss(norm, x))) <= 1e-6


def test_batch_stager_roundtrip(cuda_device):
    """staging.BatchStager: one pinned arena, one DMA per batch, double-buffered."""
    from baseboostdepth_b200.staging import BatchStager
    gen = torch.Generator().manual_seed(1)
    template = {("a", 0): torch.rand(3, 5, 7, generator=gen), "b": torch.rand(11, generator=gen), "meta": [1, 2]}
    st = BatchStager(template, cuda_device)
    assert st.nbytes >= (3 * 5 * 7 + 11) * 4
    for it in range(4):                                  # more iterations than slots
        st.host["b"].fill_(float(it))
        slot = st.upload_async()
        v = st.views(slot)
        assert torch.equal(v[("a", 0)].cpu(), template[("a", 0)])
        assert float(v["b"][0]) == float(it)
        st.release(slot)
    torch.cuda.synchronize()


def test_batch_stager_host_rewrite_is_safe(cuda_device):
    """The host rewrites the pinned views right after starting an upload (what a collate_fn does): no batch
    may arrive torn.  64 MB per batch, so a DMA is still in flight when the next fill begins; ``stager.host``
    has to hand out a different pinned arena, and wait for the DMA that last read it."""
    from baseboostdepth_b200.staging import BatchStager
    st = BatchStager({"x": torch.zeros(16 << 20)}, cuda_device)
    seen = []
    for it in range(7):
        st.host["x"].fill_(float(it + 1))
        slot = st.upload_async()
        v = st.views(slot)["x"]
        seen.append((v.min(), v.max(), float(it + 1)))
        st.release(slot)
    torch.cuda.synchronize()
    for mn, mx, want in seen:
        assert float(mn) == want and float(mx) == want, (float(mn), float(mx), want)


def test_batch_stager_8bit_frames(cuda_device):
    """8-bit frames cross PCIe as bytes and come out as the fp32 tensors ToTensor would have made
    (datasets/mono_dataset.py:55,201-203: uint8 -> float32 / 255), next to fp32 entries; odd sizes."""
    from baseboostdepth_b200.staging import BatchStager
    gen = torch.Generator().manual_seed(2)
    frame = torch.randint(0, 256, (2, 3, 37, 53), generator=gen, dtype=torch.uint8)
    ramp = torch.arange(256, dtype=torch.uint8)
    template = {("color", 0, 0): frame, "ramp": ramp, ("disp", 0): torch.rand(2, 1, 37, 53, generator=gen)}
    st = BatchStager(template, cuda_device)
    assert st.nbytes < frame.numel() * 2 + 256 * 2 + template[("disp", 0)].numel() * 4 + 1024
    for it in range(3):
        slot = st.upload_async()
        v = st.views(slot)
        assert v[("color", 0, 0)].dtype == torch.float32
        assert torch.equal(v[("color", 0, 0)].cpu(), frame.to(torch.float32).div(255))
        assert torch.equal(v["ramp"].cpu(), ramp.to(torch.float32).div(255))
        assert torch.equal(v[("disp", 0)].cpu(), template[("disp", 0)])
        st.release(slot)
    torch.cuda.synchronize()


def test_grid_sample_on_gpu(cuda_device):
    import torch.nn.functional as F
    import baseboostdepth_b200.layers as L
    gen = torch.Generator().manual_seed(31)
    img = torch.rand(3, 3, 48, 80, generator=gen).to(cuda_device)
    base = (torch.rand(3, 2, 48, 80, generator=gen) * 2.4 - 1.2).to(cuda_device)
    w = torch.rand(3, 3, 48, 80, generator=gen).to(cuda_device)
    res = []
    for fn in (lambda i, g: F.grid_sample(i, g, align_corners=True, padding_mode="border"), L.grid_sample):
        raw = base.clone().requires_grad_(True)
        out = fn(img, raw.permute(0, 2, 3, 1))
        (out * w).sum().backward()
        res.append((out.detach(), raw.grad))
    assert max_abs(res[1][0], res[0][0]) <= 1e-6
    assert max_abs(res[1][1], res[0][1]) <= 2e-5


def test_grid_sample_image_gradient_on_gpu(cuda_device):
    """Gradient w.r.t. the sampled image (trainer.py:442 under autograd) at frame size: the sorted, atomics-free gather
    against ATen's atomic scatter (1e-5 of the peak; ATen's own result varies from run to run at that level), on
    a KITTI-like warp (smooth flow plus out-of-frame margins) and bit-identical across runs."""
    import torch.nn.functional as F
    import baseboostdepth_b200.layers as L
    gen = torch.Generator().manual_seed(41)
    n, c, h, w = 4, 3, 192, 640
    ys, xs = torch.meshgrid(torch.linspace(-1, 1, h), torch.linspace(-1, 1, w), indexing="ij")
    flow = 0.08 * torch.rand(n, 2, 1, 1, generator=gen) + 0.02 * torch.randn(n, 2, h, w, generator=gen)
    base = (torch.stack([xs, ys])[None] * 1.05 + flow).to(cuda_device)
    up = (torch.rand(n, c, h, w, generator=gen) - 0.5).to(cuda_device)
    img0 = torch.rand(n, c, h, w, generator=gen).to(cuda_device)
    res = []
    for fn in (lambda i, g: F.grid_sample(i, g, align_corners=True, padding_mode="border"), L.grid_sample, L.grid_sample):
        img = img0.clone().requires_grad_(True)
        raw = base.clone().requires_grad_(True)
        (fn(img, raw.permute(0, 2, 3, 1)) * up).sum().backward()
        res.append((img.grad.clone(), raw.grad.clone()))
    assert rel_l2(res[1][0], res[0][0]) <= 1e-6, rel_l2(res[1][0], res[0][0])
    assert max_abs(res[1][0], res[0][0]) <= 1e-5 * float(res[0][0].abs().max())
    assert torch.equal(res[1][0], res[2][0])
    assert max_abs(res[1][1], res[0][1]) <= 2e-5 * max(1.0, float(res[0][1].abs().max()))


def test_step_is_cuda_graph_capturable(cuda_device):
    """include/bbd_loss.h promises graph-capturable entry points: capture loss_step + backward once,
    replay it on new input values, compare with an eager evaluation."""
    from baseboostdepth_b200.trainer import loss_step
    cfg = dict(batch=3, height=64, width=96, baselines=[2, 1, "s"], trimin=True, decomp=False)
    opt = O.default_opt(height=64, width=96, trimin=True, batch_size=3)
    gi, go, gp = make_batch(seed=8, device=cuda_device, **cfg)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in go.items()
              if k[0] in ("disp", "cam_T_cam") and v.numel()}
    static_out = {k: leaves.get(k, v) for k, v in go.items()}
    plan = plan_for(gi["ordering"], True, False, gi[("color", "s", 0)].shape[0])
    noise = {k: v.to(cuda_device) for k, v in make_noise(plan, 64, 96, seed=2).items()}

    def run():
        for p in leaves.values():
            p.grad = None
        losses = loss_step(gi, dict(static_out), opt, plan, noise=noise, num_scales=4)
        losses["loss"].backward()
        return losses["loss"]

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            run()                                  # warm-up: caches tables, weights, allocator pools
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    for p in leaves.values():
        p.grad = None
    with torch.cuda.graph(graph):
        loss_static = loss_step(gi, dict(static_out), opt, plan, noise=noise, num_scales=4)["loss"]
        loss_static.backward()
    grads_static = {k: p.grad for k, p in leaves.items()}

    # new values in the same buffers, replay, compare with eager
    with torch.no_grad():
        leaves[("disp", 0)].mul_(0.5).add_(0.02)
        gi[("color", 1, 0)].mul_(0.9)
    graph.replay()
    torch.cuda.synchronize()
    got_loss = float(loss_static)
    got = {k: g.clone() for k, g in grads_static.items()}
    want_loss = float(run())
    torch.cuda.synchronize()
    assert got_loss == want_loss
    for k, p in leaves.items():
        assert torch.equal(got[k], p.grad), k


def test_graphed_step_over_staging_slots(cuda_device):
    """graphed.GraphedLossStep: the step replayed as a CUDA graph per staging slot, batches changing on
    the host between uploads, 8-bit frames; losses and gradients equal the eager evaluation."""
    from baseboostdepth_b200.graphed import GraphedLossStep
    from baseboostdepth_b200.staging import BatchStager
    from baseboostdepth_b200.trainer import loss_step
    cfg = dict(batch=2, height=64, width=96, baselines=[1, 1], trimin=False, decomp=False)
    opt = O.default_opt(height=64, width=96, trimin=False, batch_size=2)
    gi, go, gp = make_batch(seed=9, device="cpu", **cfg)
    plan = plan_for(gi["ordering"], False, False, None)
    template = {}
    for k, v in gi.items():
        if torch.is_tensor(v):
            frame = isinstance(k, tuple) and k[0] == "color"
            template[("in",) + (k if isinstance(k, tuple) else (k,))] = (v * 255).round().to(torch.uint8) if frame else v
    for k, v in go.items():
        if k[0] in ("disp", "cam_T_cam") and v.numel():
            template[("leaf",) + k] = v.detach()
    st = BatchStager(template, cuda_device)

    def make_io(v):
        gin, gout, lv = {"ordering": gi["ordering"]}, {}, {}
        for k, t in v.items():
            if k[0] == "in":
                gin[k[1] if len(k) == 2 else k[1:]] = t
            else:
                gout[k[1:]] = lv[k[1:]] = t.detach().requires_grad_(True)
        return gin, gout, lv

    step = GraphedLossStep(st, make_io, opt, plan, num_scales=4)
    got = []
    slot = st.upload_async()
    for it in range(4):
        st.host[("leaf", "disp", 0)].mul_(0.9).add_(0.01)           # the next batch differs
        nxt = st.upload_async()
        torch.manual_seed(100 + it)                                  # noise drawn inside the graph
        step.launch(slot)
        grads = {k: g.clone() for k, g in step.grads(slot).items()}
        # eager evaluation of the same slot contents with the same noise stream
        gin, gout, lv = make_io(st.views(slot))
        torch.manual_seed(100 + it)
        want = loss_step(gin, gout, opt, plan, noise=None, num_scales=4)["loss"]
        want.backward()
        torch.cuda.synchronize()
        v = step.collect()
        if v is not None:
            got.append(v)
        for k, p in lv.items():
            assert rel_l2(grads[k], p.grad) <= 1e-6, k
        wants = float(want)
        slot = nxt
        last_want = wants
    got.append(step.collect(final=True))
    assert len(got) == 4 and abs(got[-1] - last_want) <= 2e-6


def test_sql_mode_matches_oracle(cuda_device):
    """opt.SQL: the network output is depth itself (trainer.py:457-458); single scale like the reference uses."""
    cfg = dict(batch=2, height=64, width=96, baselines=[1, 1], trimin=False, decomp=False)
    opt = O.default_opt(height=64, width=96, scales=[0], SQL=True, batch_size=2)
    inputs, outputs, params = make_batch(seed=12, device="cpu", scales=(0,), **cfg)
    with torch.no_grad():
        params[("disp", 0)].mul_(20.0).add_(1.0)          # depth-like magnitudes
    plan = plan_for(inputs["ordering"], False, False, None)
    noise = make_noise(plan, 64, 96, seed=3)
    retain_pose_grads(outputs)
    ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
    ref["loss"].backward()
    gi, go, leaves = mirror_to_device(inputs, outputs, params, cuda_device)
    losses, _ = run_fused(gi, go, opt, {k: v.to(cuda_device) for k, v in noise.items()}, 4, groups=aux["groups"])
    losses["loss"].backward()
    assert abs(float(losses["loss"]) - float(ref["loss"])) <= 2e-6
    assert rel_l2(leaves[("disp", 0)].grad, params[("disp", 0)].grad) <= 1e-5


def test_depth_planes_against_aten_cpu_and_cuda(cuda_device):
    """disparity -> depth at the benchmark size: bit-identical to the reference's ops on the CPU
    (F.interpolate + disp_to_depth, trainer.py:456-460) and within one ulp of the same ops run by ATen's
    CUDA kernels (what the reference launches on a GPU; its upsample kernel contracts differently)."""
    import ctypes as C
    import torch.nn.functional as F
    from baseboostdepth_b200 import _lib
    be = _lib.cuda_backend()
    B, H, W, S = 2, 192, 640, 4
    gen = torch.Generator().manual_seed(5)
    disps = [0.01 + 0.3 * torch.rand(B, 1, H >> s, W >> s, generator=gen) for s in range(S)]
    dev_disps = [d.to(cuda_device) for d in disps]
    a = _lib.D2DArgs()
    a.batch, a.levels, a.height, a.width = B, S, H, W
    a.min_disp, a.disp_span, a.sql = 1 / 100.0, 1 / 0.1 - 1 / 100.0, 0
    depth = torch.empty(S, B, H, W, device=cuda_device)
    for l, d in enumerate(dev_disps):
        a.h[l], a.w[l], a.disp[l] = d.shape[2], d.shape[3], d.data_ptr()
    a.depth = depth.data_ptr()
    be.call("disp_to_depth_forward", C.byref(a))
    torch.cuda.synchronize()

    def reference(d):
        up = F.interpolate(d, [H, W], mode="bilinear", align_corners=False)
        return (1 / (1 / 100.0 + (1 / 0.1 - 1 / 100.0) * up))[:, 0]

    for l in range(S):
        assert torch.equal(depth[l].cpu(), reference(disps[l])), l
        on_gpu = reference(dev_disps[l])
        rel = ((depth[l] - on_gpu).abs() / on_gpu.abs()).max().item()
        assert rel <= 2.5e-7, (l, rel)
