"""The CPU harness takes its launch decisions from the library's: for a sweep of fused-loss argument blocks both
answer the same partial-slot count, self-finalization and kernel name, and both size the smoothness and disparity
scratch alike.  The decision tests launch no compute: their argument blocks hold stand-in addresses that nothing
dereferences.

The alignment decisions are then run through the harness with buffers that start 4 bytes past a 16-byte boundary,
one at a time: the host build of every 16-byte access asserts its alignment, so a decision that lets a misaligned
vector access through aborts the run.  The last test checks that the GPU case table (tests/launch_forms.py) names
exactly the fused-loss kernels the launch description can produce."""
import ctypes as C
import itertools

import pytest
import torch

from baseboostdepth_b200 import _lib
from baseboostdepth_b200 import build as bbd_build
from baseboostdepth_b200.synthetic import make_batch, make_noise
from baseboostdepth_b200.trainer import plan_for
from fused_util import emu_backend, run_fused
from launch_forms import declared_kernel_names
from oracle import loss_path as O

B, S = 12, 4
SIZES = [(192, 640), (24, 40), (40, 70), (200, 330)]


@pytest.fixture(scope="module")
def lib():
    dll = C.CDLL(bbd_build.build())
    dll.bbd_reproj_kernel_name.restype = C.c_char_p
    dll.bbd_smooth_scratch_floats.restype = C.c_size_t
    dll.bbd_d2d_scratch_floats.restype = C.c_size_t
    return dll


@pytest.fixture(scope="module")
def emu():
    dll = emu_backend().dll
    dll.emu_reproj_kernel_name.restype = C.c_char_p
    dll.emu_smooth_scratch_floats.restype = C.c_size_t
    dll.emu_d2d_scratch_floats.restype = C.c_size_t
    return dll


@pytest.fixture(autouse=True)
def default_form(monkeypatch):
    monkeypatch.delenv("BBD_PIPE", raising=False)


POINTERS = ("target", "depth", "inv_K", "P", "ident_min", "loss_part", "gpose_part", "gdepth")


def reproj_args(H, W, max_rep, need_grad=False, winner=False, tickets=False, force_tile=False, rgba=True, offset=None):
    """Stand-in argument block; ``offset`` names one pointer ("frames_rgba" for the first copy) moved 4 bytes."""
    ra = _lib.ReprojArgs()
    ra.batch, ra.height, ra.width, ra.num_scales = B, H, W, S
    ra.need_grad, ra.max_rep, ra.min_rep, ra.num_pose, ra.force_tile = int(need_grad), max_rep, 1, 2 * B, int(force_tile)
    addr = iter(range(1 << 24, 1 << 40, 1 << 20))   # 16-byte aligned, distinct, never read
    for name in POINTERS:
        setattr(ra, name, next(addr) + (4 if name == offset else 0))
    for f in range(2):
        ra.frames[f] = next(addr)
        ra.frames_rgba[f] = (next(addr) + (4 if offset == "frames_rgba" and f == 0 else 0)) if rgba else None
    ra.winner = next(addr) if winner else None
    if tickets:
        ra.tickets, ra.pair_sum, ra.loss_out, ra.gpose_out = next(addr), next(addr), next(addr), next(addr)
    return ra


def answers(dll, prefix, ra):
    name = getattr(dll, prefix + "reproj_kernel_name")(C.byref(ra)).decode()
    if prefix == "emu_" and not torch.cuda.is_available():
        name = name.replace("_tma", "")   # without a driver the library finds no tensor-map encoder
    return (getattr(dll, prefix + "reproj_tiles")(ra.height, ra.width),
            getattr(dll, prefix + "reproj_finalizes_itself")(C.byref(ra)), name)


@pytest.mark.parametrize("max_rep", [1, 2, 3, 12])
@pytest.mark.parametrize("H,W", SIZES)
def test_reproj_decisions_agree(lib, emu, H, W, max_rep):
    for flags in itertools.product([False, True], repeat=5):
        for offset in (None,) + POINTERS + ("frames_rgba",):
            ra = reproj_args(H, W, max_rep, *flags, offset=offset)
            assert answers(lib, "bbd_", ra) == answers(emu, "emu_", ra), (flags, offset)


@pytest.mark.parametrize("offset", ["target", "depth", "ident_min"])
def test_unaligned_planes_take_plain_loads(emu, offset):
    """The TMA unit needs 16-byte aligned planes: one plane 4 bytes off selects the plain-load streaming kernel."""
    def name(ra):
        return emu.emu_reproj_kernel_name(C.byref(ra)).decode()
    assert name(reproj_args(192, 640, 2, need_grad=True, tickets=True)) == "bbd::reproj_stream_tma_kernel<2, 1, 0>"
    assert name(reproj_args(192, 640, 2, need_grad=True, tickets=True, offset=offset)) == "bbd::reproj_stream_kernel<2, 1, 0>"


def test_unaligned_rgba_copies_are_rejected(lib, emu):
    """frames_rgba entries are read and written one 16-byte pixel at a time: an entry that is not 16-byte aligned is
    an argument error (BBD_E_ARG) of bbd_reproj_fused, bbd_ident_forward and bbd_pack_rgba, before anything is
    launched or read.  The harness answers the same."""
    ra = reproj_args(64, 96, 2, need_grad=True, offset="frames_rgba")
    ia = _lib.IdentArgs()
    ia.batch, ia.height, ia.width = 2, 64, 96
    ia.target, ia.ident_min, ia.tab.hdr, ia.tab.ident = 1 << 24, 2 << 24, 3 << 24, 4 << 24
    ia.frames[0], ia.frames_rgba[0] = 5 << 24, (6 << 24) + 4
    for dll, prefix, tail in ((lib, "bbd_", (None,)), (emu, "emu_", ())):
        ra.tab.hdr, ra.tab.rep = 7 << 24, 8 << 24
        assert getattr(dll, prefix + "reproj_fused")(C.byref(ra), *tail) == -1, prefix
        assert getattr(dll, prefix + "ident_forward")(C.byref(ia), *tail) == -1, prefix
    assert lib.bbd_pack_rgba(1, 64, 96, C.c_void_p(1 << 24), C.c_void_p((2 << 24) + 4), None) == -1


# ---- alignment decisions run through the harness ----------------------------------------------------------------
def _offset(t):
    """A copy of t whose first element sits 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 4, dtype=t.dtype)
    assert buf.data_ptr() % 16 == 0
    out = buf[1:1 + t.numel()].view(t.shape)
    out.copy_(t)
    return out


def _d2d(H, W, factors, Bn=2, offset=None, seed=3):
    """(args, buffers) of a disparity -> depth call on host tensors; ``offset`` names one buffer moved 4 bytes
    ("disp0", "depth", "gdepth", "gdisp0", "gsmooth0", ...)."""
    gen = torch.Generator().manual_seed(seed)
    n = len(factors)
    t = {f"disp{l}": 0.01 + 0.3 * torch.rand(Bn, H // f, W // f, generator=gen) for l, f in enumerate(factors)}
    t.update({f"gdisp{l}": torch.zeros(Bn, H // f, W // f) for l, f in enumerate(factors)})
    t.update({f"gsmooth{l}": torch.randn(Bn, H // f, W // f, generator=gen) for l, f in enumerate(factors)})
    t["depth"], t["gdepth"] = torch.zeros(n, Bn, H, W), torch.randn(n, Bn, H, W, generator=gen)
    t["gscale"], t["gsmooth_scale"] = torch.rand(n, generator=gen), torch.rand(n, generator=gen)
    if offset:
        t[offset] = _offset(t[offset])
    a = _lib.D2DArgs()
    a.batch, a.levels, a.height, a.width = Bn, n, H, W
    a.min_disp, a.disp_span, a.sql = 1 / 100.0, 1 / 0.1 - 1 / 100.0, 0
    for l, f in enumerate(factors):
        a.h[l], a.w[l] = H // f, W // f
        a.disp[l], a.gdisp[l], a.gsmooth[l] = t[f"disp{l}"].data_ptr(), t[f"gdisp{l}"].data_ptr(), t[f"gsmooth{l}"].data_ptr()
    a.depth, a.gdepth, a.gscale, a.gsmooth_scale = (t[k].data_ptr() for k in ("depth", "gdepth", "gscale", "gsmooth_scale"))
    t["scratch"] = torch.zeros(max(1, emu_backend().value("d2d_scratch_floats", C.byref(a))))
    a.scratch = t["scratch"].data_ptr()
    return a, t


D2D_OFFSETS = [None, "disp0", "disp1", "depth", "gdepth", "gdisp0", "gdisp1", "gsmooth0"]


@pytest.mark.parametrize("offset", D2D_OFFSETS)
@pytest.mark.parametrize("H,W", [(16, 24), (12, 20)])
def test_disp_to_depth_with_unaligned_buffers(H, W, offset):
    """Disparity -> depth forward and backward through the harness, every level a 1/2/4 reduction (the single-launch
    backward when everything is aligned), with one buffer 4 bytes off.  The forms the decisions pick run without a
    misaligned 16-byte access and give what the aligned call gives: the same depth planes and the same gradient of
    the full-resolution level, bit for bit, and the coarser levels' gradients up to the summation order of the
    two-pass form."""
    factors, be = (1, 2, 4), emu_backend()
    ref, rt = _d2d(H, W, factors)
    be.call("disp_to_depth_forward", C.byref(ref))
    be.call("disp_to_depth_backward", C.byref(ref))
    a, t = _d2d(H, W, factors, offset=offset)
    be.call("disp_to_depth_forward", C.byref(a))
    be.call("disp_to_depth_backward", C.byref(a))
    assert torch.equal(t["depth"], rt["depth"])
    assert torch.equal(t["gdisp0"], rt["gdisp0"])
    for l in range(1, len(factors)):
        assert torch.allclose(t[f"gdisp{l}"], rt[f"gdisp{l}"], rtol=1e-6, atol=1e-7 * float(rt[f"gdisp{l}"].abs().max())), l


@pytest.mark.parametrize("layout", [dict(baselines=[1, 1], trimin=False), dict(baselines=[2, "s"], trimin=True)])
def test_fused_step_with_unaligned_target(layout):
    """One fused step through the harness with the target 4 bytes off a 16-byte boundary: the plain-load streaming
    form (no TMA box over an unaligned plane), bit-identical to the aligned step's TMA form, which differs only in
    how it stages three planes."""
    H, W = 24, 40
    opt = O.default_opt(height=H, width=W, scales=[0, 1], batch_size=2, **{k: v for k, v in layout.items() if k == "trimin"})
    be = emu_backend()
    got = []
    for shift in (False, True):
        inputs, outputs, params = make_batch(seed=5, batch=2, height=H, width=W, scales=(0, 1), **layout)
        if shift:
            inputs[("color", 0, 0)] = _offset(inputs[("color", 0, 0)])
            assert inputs[("color", 0, 0)].data_ptr() % 16 == 4
        plan = plan_for(inputs["ordering"], opt.trimin, False,
                        inputs[("color", "s", 0)].shape[0] if ("color", "s", 0) in inputs else None)
        losses, _ = run_fused(inputs, outputs, opt, make_noise(plan, H, W, seed=6), 4, backend=be)
        losses["loss"].backward()
        got.append((float(losses["loss"]), {k: v.grad.clone() for k, v in params.items()}, outputs["argmin"].clone()))
    assert got[0][0] == got[1][0]
    for k in got[0][1]:
        assert torch.equal(got[0][1][k], got[1][1][k]), k
    assert torch.equal(got[0][2], got[1][2])


# ---- the GPU case table names every form -------------------------------------------------------------------------
def test_gpu_table_covers_every_kernel_form(emu, monkeypatch):
    """The set of fused-loss kernels the launch description produces (for a B200 with TMA) over a sweep of sizes,
    candidate counts, flags, pointer offsets and BBD_PIPE equals the set tests/launch_forms.py declares: a new
    form cannot land without a GPU case, and the table cannot claim a form that no call reaches."""
    produced = set()
    sizes = [(192, 640), (24, 40), (50, 90), (40, 70), (16, 6152), (260, 12), (16, 16)]
    for pipe in ("0", "1"):
        monkeypatch.setenv("BBD_PIPE", pipe)
        for (H, W), max_rep in itertools.product(sizes, [1, 2, 3, 6, 12]):
            for flags in itertools.product([False, True], repeat=5):
                for offset in (None, "target", "depth", "ident_min", "frames_rgba"):
                    ra = reproj_args(H, W, max_rep, *flags, offset=offset)
                    produced.add(emu.emu_reproj_kernel_name(C.byref(ra)).decode())
    declared = declared_kernel_names()
    assert produced == declared, ("produced, not declared", sorted(produced - declared),
                                  "declared, not produced", sorted(declared - produced))


@pytest.mark.parametrize("kw,name,finalizes", [
    (dict(max_rep=2, need_grad=True, tickets=True), "bbd::reproj_stream_kernel<2, 1, 0>", 1),
    (dict(max_rep=12, need_grad=True, winner=True, tickets=True), "bbd::reproj_stream_kernel<2, 1, 1, 1>", 0),
    (dict(max_rep=12), "bbd::reproj_stream_kernel<2, 0, 1>", 0),
    (dict(max_rep=2, need_grad=True, force_tile=True), "bbd::reproj_kernel<1, 1>", 0),
])
def test_reproj_decisions_at_the_benchmark_size(lib, emu, kw, name, finalizes):
    ra = reproj_args(192, 640, **kw)
    for dll, prefix in ((lib, "bbd_"), (emu, "emu_")):
        _, fin, got = answers(dll, prefix, ra)
        assert (got.replace("_tma", ""), fin) == (name, finalizes), prefix


@pytest.mark.parametrize("H,W", SIZES)
def test_scratch_sizes_agree(lib, emu, H, W):
    levels = (C.c_int32 * _lib.MAX_SCALES)(*[H >> s for s in range(S)]), (C.c_int32 * _lib.MAX_SCALES)(*[W >> s for s in range(S)])
    assert lib.bbd_smooth_scratch_floats(B, S, *levels) == emu.emu_smooth_scratch_floats(B, S, *levels)
    da = _lib.D2DArgs()
    da.batch, da.levels, da.height, da.width = B, S, H, W
    for s in range(S):
        da.h[s], da.w[s] = H >> s, W >> s
    assert lib.bbd_d2d_scratch_floats(C.byref(da)) == emu.emu_d2d_scratch_floats(C.byref(da)) > 0
