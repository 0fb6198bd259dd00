"""Tier-A operators (drop-in ``layers`` module) against the oracle, kernels stepped on the CPU."""
import pytest
import torch

import baseboostdepth_b200.layers as L
from fused_util import emu_backend
from helpers import Golden, golden_cases, max_abs, rel_l2
from oracle import loss_path as O


@pytest.fixture(autouse=True)
def use_emulator():
    L._TEST_BACKEND = emu_backend()
    yield
    L._TEST_BACKEND = None


def _geometry(n=3, H=24, W=40, seed=0):
    g = torch.Generator().manual_seed(seed)
    K = torch.tensor([[0.58 * W, 0, 0.5 * W, 0], [0, 1.92 * H, 0.5 * H, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
    K = K.unsqueeze(0).repeat(n + 1, 1, 1)
    inv_K = torch.linalg.pinv(K)
    aa = 0.02 * torch.randn(n, 1, 3, generator=g)
    tr = 0.05 * torch.randn(n, 1, 3, generator=g)
    depth = (1.0 + 5.0 * torch.rand(n, 1, H, W, generator=g))
    return K, inv_K, aa, tr, depth


def test_backproject_project_forward_backward():
    n, H, W = 3, 24, 40
    K, inv_K, aa, tr, depth = _geometry(n, H, W)
    outs = []
    for mine in (False, True):
        d = depth.clone().requires_grad_(True)
        a, t = aa.clone().requires_grad_(True), tr.clone().requires_grad_(True)
        T = L.transformation_from_parameters(a, t)
        if mine:
            bp, pj = L.BackprojectDepth(n + 1, H, W), L.Project3D(n + 1, H, W)   # batch_size > n: sub-batch
            cam = bp(d, inv_K[:n])
            pix = pj(cam, K[:n], T)
        else:
            cam = O.backproject(d, inv_K[:n], H, W)
            pix = O.project(cam, K[:n], T, H, W)
        w = torch.linspace(0.5, 1.5, pix.numel()).view_as(pix)
        (pix * w).sum().backward()
        outs.append((cam.detach(), pix.detach(), d.grad, a.grad, t.grad))
    ref, got = outs
    assert got[1].shape == ref[1].shape and got[1].stride() == ref[1].stride()   # same non-contiguous view
    assert max_abs(got[0], ref[0]) == 0.0
    assert max_abs(got[1], ref[1]) <= 1e-6
    for i in (2, 3, 4):
        assert rel_l2(got[i], ref[i]) <= 1e-5, i


@pytest.mark.parametrize("shape", [(2, 3, 16, 20), (1, 1, 2, 5), (2, 2, 9, 3)])
def test_ssim_forward_backward(shape):
    g = torch.Generator().manual_seed(1)
    x0, y0 = torch.rand(*shape, generator=g), torch.rand(*shape, generator=g)
    w = torch.rand(*shape, generator=g)
    res = []
    for mine in (False, True):
        x, y = x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)
        out = L.SSIM()(x, y) if mine else O.ssim(x, y)
        (out * w).sum().backward()
        res.append((out.detach(), x.grad, y.grad))
    assert max_abs(res[1][0], res[0][0]) <= 1e-6
    assert rel_l2(res[1][1], res[0][1]) <= 2e-5
    assert rel_l2(res[1][2], res[0][2]) <= 2e-5


def test_ssim_accepts_non_contiguous():
    g = torch.Generator().manual_seed(2)
    x = torch.rand(2, 8, 10, 3, generator=g).permute(0, 3, 1, 2)
    y = torch.rand(2, 3, 8, 10, generator=g)
    assert max_abs(L.SSIM()(x, y), O.ssim(x, y)) <= 1e-6


def test_smooth_loss_forward_backward():
    g = torch.Generator().manual_seed(3)
    img = torch.rand(3, 3, 12, 50, generator=g)
    d0 = torch.rand(3, 1, 12, 50, generator=g)
    res = []
    for mine in (False, True):
        d = d0.clone().requires_grad_(True)
        norm = d / (d.mean(2, True).mean(3, True) + 1e-7)      # as the trainer does (trainer.py:560-562)
        loss = (L.get_smooth_loss if mine else O.smooth_loss)(norm, img)
        (2.5 * loss).backward()
        res.append((loss.detach(), d.grad))
    assert abs(float(res[1][0]) - float(res[0][0])) <= 1e-6
    assert rel_l2(res[1][1], res[0][1]) <= 1e-5


def test_module_surface():
    names = ["SSIM", "BackprojectDepth", "Project3D", "transformation_from_parameters", "disp_to_depth",
             "get_smooth_loss", "compute_depth_errors", "ConvBlock", "Conv3x3", "upsample", "rot_from_axisangle",
             "get_translation_matrix"]
    for n in names:
        assert hasattr(L, n), n
    assert len(list(L.BackprojectDepth(2, 8, 8).state_dict())) == 0      # stateless; never checkpointed
    assert len(list(L.Project3D(2, 8, 8).state_dict())) == 0
    L.SSIM().to("cpu")


def test_geometry_helpers_bit_identical():
    """Pose assembly against the oracle's element-by-element form of the reference's (layers.py:25-100);
    disp_to_depth against the depth planes the reference itself wrote into the golden cases (at scale 0 its
    upsample to the same size is a copy, so the plane is disp_to_depth of the stored disparity)."""
    g = torch.Generator().manual_seed(4)
    aa, tr = 0.3 * torch.randn(5, 1, 3, generator=g), torch.randn(5, 1, 3, generator=g)
    from baseboostdepth_b200 import geometry as G
    for inv in (False, True):
        want = O.transformation_from_parameters(aa, tr, inv)
        assert torch.equal(G.transformation_from_parameters(aa, tr, inv), want)       # tensor version
        assert max_abs(L.transformation_from_parameters(aa, tr, inv), want) <= 2e-7    # fused kernel
    for case in golden_cases():
        gc = Golden(case)
        want = gc.ref_out[("depth", 0, 0)]
        assert torch.equal(L.disp_to_depth(gc.params[("disp", 0)].detach(), 0.1, 100)[1], want), case


def test_reference_trainer_runs_unchanged_on_drop_in_layers(monkeypatch):
    """Tier A end to end: the reference's generate_images_pred + compute_losses, as oracle.loss_path restates them
    call for call, with every layers.py operator they use (and F.grid_sample, trainer.py:439,442) replaced by this
    package's drop-in, against the loss and gradients the reference itself wrote into a golden case."""
    g = Golden("plain_pm1")
    B = len(g.baselines)
    monkeypatch.setattr(O, "backproject", lambda d, inv_K, H, W: L.BackprojectDepth(B, H, W)(d, inv_K))
    monkeypatch.setattr(O, "project", lambda cam, K, T, H, W: L.Project3D(B, H, W)(cam, K, T))
    monkeypatch.setattr(O, "warp", L.grid_sample)
    monkeypatch.setattr(O, "ssim", L.SSIM())
    monkeypatch.setattr(O, "smooth_loss", L.get_smooth_loss)
    monkeypatch.setattr(O, "disp_to_depth", L.disp_to_depth)
    losses, _ = O.run(g.inputs, g.outputs, g.opt(), g.noise, num_scales=g.num_scales)
    assert abs(float(losses["loss"]) - g.losses["loss"]) <= 2e-6
    losses["loss"].backward()
    for k, ref in g.grads.items():
        assert rel_l2(g.params[k].grad, ref) <= 2e-5, k


@pytest.mark.parametrize("invert", [False, True])
def test_pose_kernel_matches_tensor_version(invert):
    from baseboostdepth_b200 import geometry as G
    gen = torch.Generator().manual_seed(11)
    aa0 = 0.3 * torch.randn(7, 1, 3, generator=gen)
    aa0[0] = 0.0                                   # zero rotation: angle = 0 is a legal network output
    tr0 = torch.randn(7, 1, 3, generator=gen)
    w = torch.randn(7, 4, 4, generator=gen)
    res = []
    for fn in (G.transformation_from_parameters, L.transformation_from_parameters):
        aa, tr = aa0.clone().requires_grad_(True), tr0.clone().requires_grad_(True)
        T = fn(aa, tr, invert)
        (T * w).sum().backward()
        res.append((T.detach(), aa.grad, tr.grad))
    assert max_abs(res[1][0], res[0][0]) <= 1e-6
    assert rel_l2(res[1][1][1:], res[0][1][1:]) <= 1e-5
    assert rel_l2(res[1][2], res[0][2]) <= 1e-5
    assert torch.isfinite(res[1][1]).all()


def test_grid_sample_matches_aten():
    import torch.nn.functional as F
    gen = torch.Generator().manual_seed(21)
    img = torch.rand(2, 3, 10, 14, generator=gen)
    base = torch.rand(2, 2, 6, 9, generator=gen) * 2.6 - 1.3          # some coordinates outside [-1, 1]
    base[0, 0, 0, 0], base[0, 1, 0, 1] = -1.0, 1.0                   # exactly on the border
    w = torch.rand(2, 3, 6, 9, generator=gen)
    res = []
    for fn in (lambda i, g: F.grid_sample(i, g, align_corners=True, padding_mode="border"), L.grid_sample):
        raw = base.clone().requires_grad_(True)
        grid = raw.permute(0, 2, 3, 1)                               # the non-contiguous view Project3D returns
        out = fn(img, grid)
        (out * w).sum().backward()
        res.append((out.detach(), raw.grad))
    assert max_abs(res[1][0], res[0][0]) <= 1e-6
    assert max_abs(res[1][1], res[0][1]) <= 1e-5


@pytest.mark.parametrize("shape", [((2, 3, 10, 14), (6, 9)), ((1, 1, 5, 4), (12, 11)), ((3, 2, 8, 8), (8, 8))])
def test_grid_sample_image_gradient_matches_aten(shape):
    """d/d(images) of grid_sample (trainer.py:442 under autograd): the sorted gather against ATen's scatter, with
    coordinates outside the frame (clamped onto the border rows / columns: long runs for one destination),
    exactly on the border, and more outputs than source pixels."""
    import torch.nn.functional as F
    (n, c, h, w), (ho, wo) = shape
    gen = torch.Generator().manual_seed(5)
    base = torch.rand(n, 2, ho, wo, generator=gen) * 2.8 - 1.4
    base[0, 0, 0, 0], base[0, 1, 0, 1] = -1.0, 1.0
    up = torch.rand(n, c, ho, wo, generator=gen) - 0.3
    res = []
    for fn in (lambda i, g: F.grid_sample(i, g, align_corners=True, padding_mode="border"), L.grid_sample):
        img = torch.rand(n, c, h, w, generator=torch.Generator().manual_seed(6)).requires_grad_(True)
        raw = base.clone().requires_grad_(True)
        out = fn(img, raw.permute(0, 2, 3, 1))
        (out * up).sum().backward()
        res.append((img.grad.clone(), raw.grad.clone()))
    assert rel_l2(res[1][0], res[0][0]) <= 1e-6, rel_l2(res[1][0], res[0][0])
    assert max_abs(res[1][0], res[0][0]) <= 1e-5 * float(res[0][0].abs().max())
    assert max_abs(res[1][1], res[0][1]) <= 1e-5
    # the image gradient alone (grid detached), and bit-reproducible
    img = torch.rand(n, c, h, w, generator=torch.Generator().manual_seed(6)).requires_grad_(True)
    a = torch.autograd.grad((L.grid_sample(img, base.permute(0, 2, 3, 1)) * up).sum(), img)[0]
    b = torch.autograd.grad((L.grid_sample(img, base.permute(0, 2, 3, 1)) * up).sum(), img)[0]
    assert torch.equal(a, b) and torch.equal(a, res[1][0])


def test_u8_to_f32_is_totensor():
    """bbd_u8_to_f32 (kernel source stepped on the CPU) == torchvision ToTensor's arithmetic for all 256 codes."""
    import ctypes
    be = emu_backend()
    src = torch.arange(256, dtype=torch.uint8).repeat(3)
    dst = torch.empty(src.numel(), dtype=torch.float32)
    be.call("u8_to_f32", ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(dst.data_ptr()), ctypes.c_size_t(src.numel()))
    assert torch.equal(dst, src.to(torch.float32).div(255))


@pytest.mark.parametrize("sizes", [((24, 40), [(24, 40), (12, 20), (6, 10), (3, 5)]),
                                   ((16, 24), [(8, 12), (2, 3)]),
                                   ((64, 96), [(64, 96), (32, 48), (16, 24), (8, 12)])])
def test_disp_to_depth_against_autograd(sizes):
    """bbd_disp_to_depth_forward/backward (and the two backward passes on their own) vs
    F.interpolate(bilinear, align_corners=False) + disp_to_depth under autograd (trainer.py:456-460)."""
    import ctypes as C
    import torch.nn.functional as F
    from baseboostdepth_b200 import _lib
    be = emu_backend()
    (H, W), levels = sizes
    B, S = 2, len(levels)
    gen = torch.Generator().manual_seed(3)
    disps = [(0.01 + 0.3 * torch.rand(B, 1, h, w, generator=gen)).requires_grad_(True) for h, w in levels]
    gdepth = torch.randn(S, B, H, W, generator=gen)
    gscale = torch.rand(S, generator=gen) + 0.5
    min_disp, span = 1 / 100.0, 1 / 0.1 - 1 / 100.0

    want_depth, want_grads = [], []
    for l, d in enumerate(disps):
        up = F.interpolate(d, [H, W], mode="bilinear", align_corners=False)
        depth = 1 / (min_disp + span * up)
        want_depth.append(depth.detach()[:, 0])
        (depth[:, 0] * gdepth[l] * gscale[l]).sum().backward()
        want_grads.append(d.grad.clone())

    a = _lib.D2DArgs()
    a.batch, a.levels, a.height, a.width = B, S, H, W
    a.min_disp, a.disp_span, a.sql = min_disp, span, 0
    depth = torch.empty(S, B, H, W)
    cont = [d.detach().contiguous() for d in disps]
    for l, d in enumerate(cont):
        a.h[l], a.w[l], a.disp[l] = d.shape[2], d.shape[3], d.data_ptr()
    a.depth = depth.data_ptr()
    be.call("disp_to_depth_forward", C.byref(a))
    for l in range(S):
        # ATen's CPU upsample has two code paths: from 64x96 outputs on (the sizes that matter) the kernel
        # reproduces it bit for bit; for tiny outputs ATen rounds its lerps differently by one ulp
        if H * W >= 64 * 96:
            assert torch.equal(depth[l], want_depth[l]), l
        else:
            assert float(((depth[l] - want_depth[l]).abs() / want_depth[l].abs()).max()) <= 5e-7, l

    def backward(split):
        out = [torch.full_like(d, float("nan")) for d in cont]
        a.gdepth, a.gscale = gdepth.data_ptr(), gscale.data_ptr()
        for l, g in enumerate(out):
            a.gdisp[l] = g.data_ptr()
        scratch = torch.empty(max(1, be.value("d2d_scratch_floats", C.byref(a))))
        a.scratch = scratch.data_ptr()
        if split:
            be.call("disp_to_depth_backward_pass2", C.byref(a), 0, 1)   # a full-resolution level needs no pass 1
            be.call("disp_to_depth_backward_pass1", C.byref(a))
            be.call("disp_to_depth_backward_pass2", C.byref(a), 1, S)
        else:
            be.call("disp_to_depth_backward", C.byref(a))
        return out

    whole = backward(False)
    for l in range(S):
        assert rel_l2(whole[l], want_grads[l]) <= 2e-6, (l, rel_l2(whole[l], want_grads[l]))
    if levels[0] == (H, W):
        parts = backward(True)
        for l in range(S):
            # the single-launch form adds the window column-first, the two passes row-first: same terms, other order
            assert rel_l2(parts[l], whole[l]) <= 2e-6, l
            assert rel_l2(parts[l], want_grads[l]) <= 2e-6, l


def test_operator_size_sweep():
    """Tier-A operators over a sweep of small and awkward sizes (2-pixel images, single rows of tiles, widths
    around the 28-column tile and the 32-lane pitch): SSIM, smoothness and grid_sample vs the ATen ops."""
    import torch.nn.functional as F
    gen = torch.Generator().manual_seed(99)
    sizes = [(2, 2), (2, 7), (3, 28), (5, 29), (4, 31), (6, 32), (7, 33), (17, 57), (16, 56), (33, 5)]
    for H, W in sizes:
        x0, y0 = torch.rand(1, 3, H, W, generator=gen), torch.rand(1, 3, H, W, generator=gen)
        w = torch.rand(1, 3, H, W, generator=gen)
        got, ref = [], []
        for mine, res in ((True, got), (False, ref)):
            x = x0.clone().requires_grad_(True)
            out = L.SSIM()(x, y0) if mine else O.ssim(x, y0)
            (out * w).sum().backward()
            res.extend([out.detach(), x.grad])
        assert max_abs(got[0], ref[0]) <= 1e-6, ("ssim", H, W)
        assert rel_l2(got[1], ref[1]) <= 5e-5, ("ssim grad", H, W, rel_l2(got[1], ref[1]))

        d0 = 0.05 + torch.rand(1, 1, H, W, generator=gen)
        got, ref = [], []
        for mine, res in ((True, got), (False, ref)):
            d = d0.clone().requires_grad_(True)
            loss = (L.get_smooth_loss if mine else O.smooth_loss)(d, x0)
            loss.backward()
            res.extend([loss.detach(), d.grad])
        assert abs(float(got[0]) - float(ref[0])) <= 1e-6, ("smooth", H, W)
        assert rel_l2(got[1], ref[1]) <= 1e-5, ("smooth grad", H, W)

        base = torch.rand(1, 2, H, W, generator=gen) * 2.4 - 1.2
        got, ref = [], []
        for fn, res in ((L.grid_sample, got),
                        (lambda i, g: F.grid_sample(i, g, align_corners=True, padding_mode="border"), ref)):
            raw = base.clone().requires_grad_(True)
            out = fn(x0, raw.permute(0, 2, 3, 1))
            (out * w).sum().backward()
            res.extend([out.detach(), raw.grad])
        assert max_abs(got[0], ref[0]) <= 1e-6, ("grid_sample", H, W)
        assert max_abs(got[1], ref[1]) <= 2e-5, ("grid_sample grad", H, W)
