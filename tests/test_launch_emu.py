"""The CPU harness takes its launch decisions from the library's: for a sweep of fused-loss argument blocks both
answer the same partial-slot count, self-finalization and kernel name, and both size the smoothness and disparity
scratch alike.  No compute is launched: the argument blocks hold stand-in addresses that nothing dereferences."""
import ctypes as C
import itertools

import pytest
import torch

from baseboostdepth_b200 import _lib
from baseboostdepth_b200 import build as bbd_build
from fused_util import emu_backend

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


def reproj_args(H, W, max_rep, need_grad=False, winner=False, tickets=False, force_tile=False, rgba=True):
    ra = _lib.ReprojArgs()
    ra.batch, ra.height, ra.width, ra.num_scales = B, H, W, S
    ra.need_grad, ra.max_rep, ra.min_rep, ra.num_pose, ra.force_tile = int(need_grad), max_rep, 1, 2 * B, int(force_tile)
    addr = iter(range(1 << 24, 1 << 40, 1 << 20))   # 16-byte aligned, distinct, never read
    for name in ("target", "depth", "inv_K", "P", "ident_min", "loss_part", "gpose_part", "gdepth"):
        setattr(ra, name, next(addr))
    for f in range(2):
        ra.frames[f] = next(addr)
        ra.frames_rgba[f] = next(addr) if rgba else None
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
        ra = reproj_args(H, W, max_rep, *flags)
        assert answers(lib, "bbd_", ra) == answers(emu, "emu_", ra), flags


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
