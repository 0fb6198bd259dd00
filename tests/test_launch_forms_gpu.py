"""Every launch form of the loss kernels on the B200, reached as production reaches it, against the oracle.

Each row of tests/launch_forms.py runs one step of ``trainer.loss_step``.  The step proves it reached its form
twice: by the kernel name the library reports for the call (exact template arguments) and by a ``torch.profiler``
trace of the step (kernel families, and no ``reproj_finalize_kernel`` where the call finalizes itself).  Then,
against the oracle on the same CPU batch: each loss within 2e-6, the selections wherever the oracle's margin exceeds
1e-6, the disparity and pose gradients (and, on a subset, every colour frame's gradient) to the parity bar of
helpers.assert_grad_parity.  A second run of the step must give bit-identical results.

Cross-form checks need no oracle: the plain-load and TMA streaming kernels differ only in how three planes are
staged, so they agree bit for bit; and the tile form's depth and argmin planes are held to the reference's on every
golden case (DESIGN.md 3).
"""
import ctypes as C
import re

import pytest
import torch
import torch.nn.functional as F

from baseboostdepth_b200 import _lib, fused
from baseboostdepth_b200.synthetic import WORKLOADS, make_batch, make_noise
from baseboostdepth_b200.trainer import loss_step, plan_for
from frame_grad_util import frame_grad, frame_keys, referenced_rows, require_frame_grads
from fused_util import mirror_to_device, retain_pose_grads
from helpers import PARITY_LOG, Golden, assert_grad_parity, golden_cases, rel_l2, selection_check
from launch_forms import CASES, Case
from oracle import loss_path as O

pytestmark = pytest.mark.gpu


# ---- batches ---------------------------------------------------------------------------------------------------
def build(case: Case, dtype=torch.float32):
    """(inputs, outputs, params, opt, plan, noise) on the CPU.  A disparity pyramid with other factors than 2**s
    (``case.factors``) and its colour levels are built here from the same seeded draws."""
    H, W = case.hw
    lay = case.layout
    scales = list(case.scales)
    cfg = dict(batch=len(lay["baselines"]), height=H, width=W, baselines=list(lay["baselines"]), trimin=lay["trimin"],
               decomp=False)
    inputs, outputs, params = make_batch(seed=case.seed, scales=(0,) if case.factors else scales, dtype=dtype, **cfg)
    if case.factors:
        gen = torch.Generator().manual_seed(case.seed + 1)
        color0 = inputs[("color", 0, 0)]
        for s, f in zip(scales, case.factors):
            if s == 0:
                continue
            inputs[("color", 0, s)] = F.avg_pool2d(color0, f)
            d = (0.01 + 0.29 * torch.rand(cfg["batch"], 1, H // f, W // f, generator=gen)).to(dtype).requires_grad_(True)
            params[("disp", s)] = outputs[("disp", s)] = d
    opt = O.default_opt(height=H, width=W, trimin=lay["trimin"], decomp=False, pose_error=5.5, scales=scales,
                        batch_size=cfg["batch"])
    plan = plan_for(inputs["ordering"], opt.trimin, False,
                    inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
    noise = make_noise(plan, H, W, seed=case.seed + 2)
    if dtype != torch.float32:
        noise = {k: v.to(dtype) for k, v in noise.items()}
    return inputs, outputs, params, opt, plan, noise


def offset_copy(t):
    """A copy of t on the same device whose first element sits 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 4, device=t.device, dtype=t.dtype)
    out = buf[1:1 + t.numel()].view(t.shape)
    out.copy_(t)
    assert out.data_ptr() % 16 == 4
    return out


class NoWinnerBackend:
    """The CUDA library as a C caller sees it that passes ``winner = NULL`` to the fused loss (and so to the
    finalize and the name query, which must describe the same launches)."""

    def __init__(self, be):
        self._be = be
        self.dll = self   # fused.py asks be.dll.bbd_reproj_kernel_name

    def __getattr__(self, name):
        return getattr(self._be, name)

    @staticmethod
    def _strip(args):
        out = []
        for a in args:
            obj = getattr(a, "_obj", None)
            if isinstance(obj, _lib.ReprojArgs):
                c = _lib.ReprojArgs.from_buffer_copy(obj)
                c.winner = None
                a = C.byref(c)
            out.append(a)
        return out

    def call(self, name, *args):
        return self._be.call(name, *self._strip(args))

    def value(self, name, *args):
        return self._be.value(name, *self._strip(args))

    def bbd_reproj_kernel_name(self, ref):
        return self._be.dll.bbd_reproj_kernel_name(*self._strip([ref]))


@pytest.fixture
def switches(monkeypatch):
    """Sets a case's switches for one test; monkeypatch restores them (and removes BBD_PIPE) afterwards."""
    def apply(case: Case):
        monkeypatch.setattr(fused, "_FORCE_TILE", case.force_tile)
        monkeypatch.setattr(fused, "_SPLIT_D2D_BACKWARD", case.split)
        monkeypatch.setattr(fused, "_USE_SIDE", case.side)
        monkeypatch.setenv("BBD_PIPE", "1" if case.pipe else "0")
    return apply


def kernel_families(prof):
    """Names (without namespace and template arguments) of the bbd kernels a profiled region launched."""
    fams = []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        m = re.search(r"bbd::(\w+)", e.name)
        if m:
            fams.append(m.group(1))
    return fams


def gpu_step(case: Case, inputs, outputs, params, opt, plan, noise, device, frame_keys_=(), profile=False):
    """One production step on the device: returns (losses, leaves, argmin or None, reported kernel name, kernel
    families or None, {frame key: gradient})."""
    gi, go, leaves = mirror_to_device(inputs, outputs, params, device)
    if case.offset_target:
        gi[("color", 0, 0)] = offset_copy(gi[("color", 0, 0)])
    for k in frame_keys_:
        gi[k] = gi[k].detach().clone() if not (case.offset_target and k == ("color", 0, 0)) else gi[k].detach()
        gi[k].requires_grad_(True)
    gnoise = {k: v.to(device) for k, v in noise.items()}
    be = _lib.cuda_backend()
    if case.no_winner:
        be = NoWinnerBackend(be)
    timers = {}
    prof = None

    def run():
        with torch.set_grad_enabled(case.grad):
            losses = loss_step(gi, go, opt, plan, noise=gnoise, num_scales=4, backend=be,
                               want_winner=not case.no_winner, timers=timers)
            if case.grad:
                losses["loss"].backward()
        torch.cuda.synchronize()
        return losses

    if profile:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            losses = run()
    else:
        losses = run()
    argmin = None if case.no_winner else go["argmin"].clone()
    fgrads = {k: frame_grad(gi, k).detach().cpu() for k in frame_keys_}
    return (losses, leaves, argmin, timers.get("reproj_kernel_name"),
            kernel_families(prof) if prof is not None else None, fgrads)


def check_form(case: Case, name, fams):
    assert name == case.reproj, (case.name, name)
    launched = set(fams)
    assert case.reproj_family in launched, (case.name, sorted(launched))
    others = {"reproj_kernel", "reproj_stream_kernel", "reproj_stream_tma_kernel", "reproj_pipe_kernel"} - {case.reproj_family}
    assert not others & launched, (case.name, sorted(launched))
    assert case.ident in launched and not ({"ident_kernel", "ident_stream_kernel"} - {case.ident}) & launched, sorted(launched)
    assert ("reproj_finalize_kernel" in launched) == case.finalize, (case.name, sorted(launched))
    d2d_all = {"d2d_backward_fused_kernel", "d2d_hpass_kernel", "d2d_backward_kernel"}
    want_d2d = set(case.d2d) if case.grad else set()
    assert launched & d2d_all == want_d2d, (case.name, sorted(launched & d2d_all))
    if case.split:
        assert fams.count("d2d_backward_kernel") == 2, fams   # the full-resolution level on its own, then the rest


def oracle(case: Case, frame_grads=False):
    inputs, outputs, params, opt, plan, noise = build(case)
    keys = frame_keys(inputs) if frame_grads else []
    require_frame_grads(inputs, keys)
    retain_pose_grads(outputs)
    with torch.set_grad_enabled(case.grad):
        ref, aux = O.run(inputs, outputs, opt, noise, num_scales=4)
        if case.grad:
            ref["loss"].backward()
    return inputs, outputs, params, opt, plan, noise, ref, aux, keys


def oracle64(case: Case, keys):
    i64, o64, p64, opt, _, noise = build(case, torch.float64)
    require_frame_grads(i64, keys)
    retain_pose_grads(o64)
    O.run(i64, o64, opt, noise, num_scales=4)[0]["loss"].backward()
    return i64, o64, p64


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_launch_form_against_oracle(case, cuda_device, switches):
    switches(case)
    inputs, outputs, params, opt, plan, noise, ref, aux, keys = oracle(case, case.frame_grads)
    fresh = build(case)
    losses, leaves, argmin, name, fams, fgrads = gpu_step(case, *fresh[:3], opt, plan, noise, cuda_device, keys,
                                                          profile=True)
    check_form(case, name, fams)
    for k in ref:
        assert abs(float(losses[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), (k, float(losses[k]),
                                                                                              float(ref[k]))
    if argmin is not None:
        selection_check(argmin, plan, aux, list(case.scales))
    r64 = None
    if case.grad:
        for k, leaf in leaves.items():
            want = params[k].grad if k[0] == "disp" else outputs[k].grad
            if rel_l2(leaf.grad, want) > 1e-5 and r64 is None:
                r64 = oracle64(case, keys)
            want64 = None if r64 is None else (r64[2][k].grad if k[0] == "disp" else r64[1][k].grad)
            assert_grad_parity(leaf.grad, want, want64, k, case="launch_forms/" + case.name)
        used = referenced_rows(plan)
        for k in keys:
            mine, want = fgrads[k], frame_grad(inputs, k)
            if rel_l2(mine, want) > 1e-5 and r64 is None:
                r64 = oracle64(case, keys)
            assert_grad_parity(mine, want, None if r64 is None else frame_grad(r64[0], k), k,
                               case="launch_forms/" + case.name)
            if k[2] == 0 and k[1] != 0:
                for r in range(mine.shape[0]):
                    if k[1] not in used or r not in used[k[1]]:
                        assert float(mine[r].abs().max()) == 0.0, (k, r)

    # determinism: the same step again, bit for bit
    again = gpu_step(case, *build(case)[:3], opt, plan, noise, cuda_device, keys)
    for k in losses:
        assert torch.equal(losses[k].detach().cpu(), again[0][k].detach().cpu()), k
    if case.grad:
        for k in leaves:
            assert torch.equal(leaves[k].grad.cpu(), again[1][k].grad.cpu()), k
    if argmin is not None:
        assert torch.equal(argmin, again[2])
    for k in keys:
        assert torch.equal(fgrads[k], again[5][k]), k


PAIRS = ["stream_k2_grad", "stream_k1_grad", "multi_grad", "multi_fwd", "stream_k2_fwd"]


@pytest.mark.parametrize("tma_case", PAIRS)
def test_plain_loads_bit_identical_to_tma(tma_case, cuda_device, switches):
    """The plain-load streaming kernel (reached here by an unaligned target) and the TMA kernel on the same batch:
    same losses, gradients and winner planes, bit for bit."""
    from launch_forms import BY_NAME
    import dataclasses
    tma = BY_NAME[tma_case]
    plain = dataclasses.replace(tma, name=tma.name + "_unaligned", offset_target=True,
                                reproj=tma.reproj.replace("_tma", ""))
    got = []
    for case in (tma, plain):
        switches(case)
        inputs, outputs, params, opt, plan, noise = build(case)
        res = gpu_step(case, inputs, outputs, params, opt, plan, noise, cuda_device)
        assert res[3] == case.reproj, res[3]
        got.append(res)
    (l0, g0, w0, _, _, _), (l1, g1, w1, _, _, _) = got
    for k in l0:
        assert torch.equal(l0[k].detach().cpu(), l1[k].detach().cpu()), k
    if tma.grad:
        for k in g0:
            assert torch.equal(g0[k].grad.cpu(), g1[k].grad.cpu()), k
    assert torch.equal(w0, w1)


@pytest.mark.parametrize("case", golden_cases())
def test_tile_form_on_golden_cases(case, cuda_device, monkeypatch):
    """The tile form ("exact mode", DESIGN.md 3) on every golden case.  Depth planes at the frame's own resolution
    equal the reference's bit for bit; the upsampled levels differ from ATen's CPU upsample by at most 4 ulp (ATen's
    CPU kernel rounds differently at these small sizes than at the benchmark size, where
    test_gpu_parity.test_depth_planes_against_aten_cpu_and_cuda holds them bit-identical; the parity log counts the
    pixels).  Argmin planes equal the fp32 oracle's everywhere, without the near-tie margin."""
    monkeypatch.setattr(fused, "_FORCE_TILE", True)
    g = Golden(case)
    ref, aux = O.run(g.inputs, g.outputs, g.opt(), g.noise, num_scales=g.num_scales)
    h = Golden(case)
    hi, ho, _ = mirror_to_device(h.inputs, h.outputs, h.params, cuda_device)
    timers = {}
    plan = plan_for(hi["ordering"], g.opt().trimin, g.opt().decomp,
                    hi[("color", "s", 0)].shape[0] if ("color", "s", 0) in hi else None, aux["groups"])
    with torch.no_grad():
        losses = loss_step(hi, ho, h.opt(), plan, noise={k: v.to(cuda_device) for k, v in h.noise.items()},
                           num_scales=h.num_scales, want_winner=True, timers=timers)
    torch.cuda.synchronize()
    assert timers["reproj_kernel_name"].startswith("bbd::reproj_kernel<0, "), timers["reproj_kernel_name"]
    for k, v in g.losses.items():
        assert abs(float(losses[k]) - v) <= 2e-6 * max(1.0, abs(v)), k
    eps = torch.finfo(torch.float32).eps
    for s in h.scales:
        mine, want = ho[("depth", 0, s)].cpu(), g.ref_out[("depth", 0, s)]
        if tuple(g.outputs[("disp", s)].shape[-2:]) == (g.H, g.W):
            assert torch.equal(mine, want), s
        ulps = float(((mine.double() - want.double()).abs() / (eps * want.double().abs())).max())
        PARITY_LOG.append({"case": "tile/" + case, "key": f"depth plane {s}", "pixels": want.numel(),
                           "pixels_not_bit_identical": int((mine != want).sum()), "max_rel_diff_in_eps": ulps})
        assert ulps <= 4.0, (s, ulps)
    selection_check(ho["argmin"], plan, aux, h.scales, exact=True)


def test_tile_form_full_size(cuda_device, switches):
    """The tile form at the benchmark size: 13k blocks and a partial-slot layout that no small case reaches."""
    batch, H, W, baselines, trimin, decomp = WORKLOADS["kitti_640x192_b12_pm1"]
    case = Case("tile_full_size", dict(baselines=list(baselines), trimin=trimin), (H, W), "bbd::reproj_kernel<1, 1>",
                finalize=True, force_tile=True, seed=1234)
    switches(case)
    inputs, outputs, params, opt, plan, noise, ref, aux, _ = oracle(case)
    losses, leaves, argmin, name, fams, _ = gpu_step(case, *build(case)[:3], opt, plan, noise, cuda_device,
                                                     profile=True)
    check_form(case, name, fams)
    for k in ref:
        assert abs(float(losses[k]) - float(ref[k])) <= 2e-6 * max(1.0, abs(float(ref[k]))), k
    selection_check(argmin, plan, aux, list(case.scales))
    r64 = None
    for k, leaf in leaves.items():
        want = params[k].grad if k[0] == "disp" else outputs[k].grad
        if rel_l2(leaf.grad, want) > 1e-5 and r64 is None:
            r64 = oracle64(case, [])
        want64 = None if r64 is None else (r64[2][k].grad if k[0] == "disp" else r64[1][k].grad)
        assert_grad_parity(leaf.grad, want, want64, k, case="launch_forms/" + case.name)
