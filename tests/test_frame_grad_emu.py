"""Gradients of the fused loss w.r.t. the colour frames, kernel source stepped on the CPU vs the oracle.

The oracle is plain ATen under autograd: setting requires_grad on the colour inputs gives the reference's
frame gradients (fp32, and fp64 as the yardstick where fp32 rounding of the reference itself misses the bar).
"""
import ctypes as C
import os
import subprocess
import tempfile

import pytest
import torch

from baseboostdepth_b200 import _lib
from baseboostdepth_b200 import layers as L
from frame_grad_util import frame_grad, frame_keys, referenced_rows, require_frame_grads
from fused_util import emu_backend, run_fused
from helpers import Golden, assert_grad_parity, golden_cases, rel_l2
from oracle import loss_path as O

CASES = golden_cases()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle_frame_grads(case, keys, dtype=torch.float32):
    g = Golden(case, dtype=dtype)
    require_frame_grads(g.inputs, keys)
    ref, aux = O.run(g.inputs, g.outputs, g.opt(), g.noise, num_scales=g.num_scales)
    ref["loss"].backward()
    return {k: frame_grad(g.inputs, k) for k in keys}, ref, aux


def _fused(case, keys, groups, detach_params=False, backend=None):
    h = Golden(case)
    if detach_params:
        for k, v in list(h.outputs.items()):
            h.outputs[k] = v.detach()
    require_frame_grads(h.inputs, keys)
    losses, plan = run_fused(h.inputs, h.outputs, h.opt(), h.noise, h.num_scales, backend=backend or emu_backend(),
                             groups=groups)
    losses["loss"].backward()
    return h, losses, plan


def check_frame_grads(case, keys, detach_params=False, backend=None, log_case=None):
    """Frame gradients of `keys` vs the oracle; rows no candidate reads exactly zero.  Returns the fused run."""
    ref32, ref, aux = _oracle_frame_grads(case, keys)
    h, losses, plan = _fused(case, keys, aux["groups"], detach_params, backend)
    for k, v in ref.items():
        assert abs(float(losses[k]) - float(v)) <= 2e-6 * max(1.0, abs(float(v))), k
    ref64 = None
    used = referenced_rows(plan)
    for k in keys:
        mine = frame_grad(h.inputs, k)
        assert mine.shape == h.inputs[k].shape, k
        if rel_l2(mine, ref32[k]) > 1e-5 and ref64 is None:
            ref64, _, _ = _oracle_frame_grads(case, keys, torch.float64)
        assert_grad_parity(mine, ref32[k], None if ref64 is None else ref64[k], k, case=log_case or case)
        f = k[1]
        if k[2] == 0 and f != 0:
            for r in range(mine.shape[0]):
                if f not in used or r not in used[f]:
                    assert float(mine[r].abs().max()) == 0.0, (k, r)
    return h, losses, plan


@pytest.mark.parametrize("case", CASES)
def test_frame_grads_match_oracle(case):
    keys = frame_keys(Golden(case).inputs)
    h, losses, _ = check_frame_grads(case, keys)
    # the disparity / pose gradients of the same step are those of the step whose frames need none
    g0 = Golden(case)
    ref, aux = O.run(g0.inputs, g0.outputs, g0.opt(), g0.noise, num_scales=g0.num_scales)
    n = Golden(case)
    losses0, _ = run_fused(n.inputs, n.outputs, n.opt(), n.noise, n.num_scales, backend=emu_backend(), groups=aux["groups"])
    losses0["loss"].backward()
    for k in losses0:
        assert torch.equal(losses0[k].detach(), losses[k].detach()), k
    for k, v in n.params.items():
        if v.grad is not None:
            assert torch.equal(v.grad, h.params[k].grad), k


@pytest.mark.parametrize("case", ["plain_pm1", "trimin_decomp"])
def test_only_the_target(case):
    check_frame_grads(case, [("color", 0, 0)])


def test_only_one_source_stack():
    check_frame_grads("trimin_mixed", [("color", -1, 0)])


@pytest.mark.parametrize("case", ["plain_mixed_s", "ragged_decomp_24x40"])
def test_frames_only_without_depth_or_pose_gradients(case):
    h, losses, _ = check_frame_grads(case, frame_keys(Golden(case).inputs), detach_params=True)
    assert all(v.grad is None for v in h.params.values())


def test_no_ssim():
    assert Golden("plain_nossim").no_ssim
    check_frame_grads("plain_nossim", frame_keys(Golden("plain_nossim").inputs))


def test_frame_grads_are_deterministic():
    keys = frame_keys(Golden("trimin_decomp").inputs)
    a, _, _ = _fused("trimin_decomp", keys, None)
    b, _, _ = _fused("trimin_decomp", keys, None)
    for k in keys:
        assert torch.equal(frame_grad(a.inputs, k), frame_grad(b.inputs, k)), k


NEW_CALLS = {"frame_grad", "frame_grad_stacks", "smooth_image_grad"}


class _Recorder:
    """Backend wrapper that records the names of the C-ABI calls of a step."""

    def __init__(self, be):
        self.be, self.names = be, []

    def __getattr__(self, name):
        return getattr(self.be, name)

    def call(self, name, *args):
        self.names.append(name)
        return self.be.call(name, *args)


@pytest.mark.parametrize("case,finalize", [("plain_pm1", []), ("trimin_decomp", ["reproj_finalize"])])
def test_default_step_makes_the_same_calls(case, finalize):
    """A step whose frames need no gradient makes exactly the calls it made before frame gradients existed
    (the fused finalize of the one/two-candidate streaming kernel saves reproj_finalize)."""
    g = Golden(case)
    rec = _Recorder(emu_backend())
    losses, _ = run_fused(g.inputs, g.outputs, g.opt(), g.noise, g.num_scales, backend=rec)
    losses["loss"].backward()
    assert rec.names == ["disp_to_depth_forward", "smooth_fused", "pose_pack_forward", "ident_forward",
                         "reproj_fused"] + finalize + ["loss_combine_forward", "loss_combine_backward",
                                                       "disp_to_depth_backward", "pose_pack_backward"], rec.names
    h = Golden(case)
    require_frame_grads(h.inputs)
    rec = _Recorder(emu_backend())
    losses, _ = run_fused(h.inputs, h.outputs, h.opt(), h.noise, h.num_scales, backend=rec)
    losses["loss"].backward()
    assert NEW_CALLS <= set(rec.names)


@pytest.mark.parametrize("shape", [(2, 3, 10, 14), (1, 3, 7, 2), (3, 3, 2, 9), (2, 3, 13, 11)])
def test_tier_a_smooth_loss_image_gradient(shape, monkeypatch):
    monkeypatch.setattr(L, "_TEST_BACKEND", emu_backend())
    gen = torch.Generator().manual_seed(17)
    n, c, h, w = shape
    disp0 = torch.rand(n, 1, h, w, generator=gen)
    img0 = torch.rand(n, c, h, w, generator=gen)
    res = []
    for fn in (O.smooth_loss, L.get_smooth_loss):
        d, im = disp0.clone().requires_grad_(True), img0.clone().requires_grad_(True)
        (fn(d, im) * 0.7).backward()
        res.append((d.grad, im.grad))
    assert rel_l2(res[1][1], res[0][1]) <= 1e-5, rel_l2(res[1][1], res[0][1])
    assert rel_l2(res[1][0], res[0][0]) <= 1e-5


def test_abi_argument_errors():
    from baseboostdepth_b200 import build as bbd_build
    dll = C.CDLL(bbd_build.build())
    null = C.c_void_p(None)
    assert dll.bbd_frame_grad(null, null, null) == -1
    assert dll.bbd_frame_grad_stacks(null, null, null) == -1
    assert dll.bbd_smooth_image_grad(null, null) == -1
    ra, fa = _lib.ReprojArgs(), _lib.FrameGradArgs()
    buf = (C.c_float * 4)()
    tab = (C.c_int32 * 64)()
    p = C.cast(buf, C.c_void_p).value
    for name in ("target", "depth", "inv_K", "P", "winner"):
        setattr(ra, name, p)
    ra.tab.hdr = ra.tab.rep = ra.tab.ident = C.cast(tab, C.c_void_p).value
    fa.gpred = fa.gident = fa.gscale = fa.keys = fa.coef = p
    ra.batch, ra.height, ra.width, ra.num_scales, ra.max_rep = 1, 32, 64, 1, 0
    assert dll.bbd_frame_grad(C.byref(ra), C.byref(fa), null) == -2
    ra.max_rep = _lib.MAX_REP + 1
    assert dll.bbd_frame_grad(C.byref(ra), C.byref(fa), null) == -2
    ra.max_rep, ra.num_scales = 2, _lib.MAX_SCALES + 1
    assert dll.bbd_frame_grad(C.byref(ra), C.byref(fa), null) == -2
    ra.num_scales, ra.height = 1, 1
    assert dll.bbd_frame_grad(C.byref(ra), C.byref(fa), null) == -1
    ra.height = 32
    fa.stack_rows[0] = -1
    assert dll.bbd_frame_grad_stacks(C.byref(ra), C.byref(fa), null) == -2
    fa.stack_rows[0] = 1
    assert dll.bbd_frame_grad_stacks(C.byref(ra), C.byref(fa), null) == -1     # sorted keys / order missing
    fa.coef = None
    assert dll.bbd_frame_grad(C.byref(ra), C.byref(fa), null) == -1            # SSIM needs the coefficient scratch
    sa = _lib.SmoothImgArgs()
    sa.gscale, sa.batch, sa.levels = p, 1, _lib.MAX_SCALES + 1
    assert dll.bbd_smooth_image_grad(C.byref(sa), null) == -2
    sa.levels = 1
    sa.gimg[0], sa.h[0], sa.w[0] = p, 1, 8
    assert dll.bbd_smooth_image_grad(C.byref(sa), null) == -1


def test_new_struct_layouts_match_header():
    src = ('#include "bbd_loss.h"\n#include <stdio.h>\nint main(){printf("%zu %zu", sizeof(bbd_frame_grad_args),'
           'sizeof(bbd_smooth_img_args));return 0;}')
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        sizes = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [C.sizeof(_lib.FrameGradArgs), C.sizeof(_lib.SmoothImgArgs)]
