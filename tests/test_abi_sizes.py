"""Size checks of the C ABI's per-pixel entry points (include/bbd_loss.h): a negative count, channel count or
size is BBD_E_ARG, an H*W / Ho*Wo / n*channels beyond int32 is BBD_E_RANGE, n == 0 is a no-op returning 0.

Each call runs in a child process that sees no GPU (CUDA_VISIBLE_DEVICES=""): a check that is missing lets the
call go on to a launch, which then fails with a CUDA error code (> 0) instead of reaching a device with a
wrapped element count.  The pointers are host scratch memory; a correct check returns before any of them is
used."""
import json
import os
import subprocess
import sys

import pytest

from baseboostdepth_b200 import build as bbd_build

E_ARG, E_RANGE = -1, -2

_CHILD = r"""
import ctypes, json, sys
lib = ctypes.CDLL(sys.argv[1])
lib.bbd_last_error_string.restype = ctypes.c_char_p
buf = ctypes.create_string_buffer(4096)
p = ctypes.c_void_p((ctypes.addressof(buf) + 15) // 16 * 16)
conv = {"p": p, "eps": ctypes.c_float(1e-7)}
args = [conv[a] if isinstance(a, str) else ctypes.c_int32(a) for a in json.loads(sys.argv[3])]
rc = getattr(lib, sys.argv[2])(*args, ctypes.c_void_p(None))
print(json.dumps({"rc": rc, "msg": lib.bbd_last_error_string().decode()}))
"""


@pytest.fixture(scope="module")
def lib_path():
    return os.environ.get("BBD_LIB") or bbd_build.build()


def call_without_gpu(lib_path, name, args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _CHILD, lib_path, name, json.dumps(args)], env=env,
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    return json.loads(res.stdout.strip().splitlines()[-1])


# (entry point, arguments before the stream) per size layout of the tier-A calls
CALLS = {
    "backproject_forward": lambda n, c, h, w, ho, wo: ("bbd_backproject_forward", [n, h, w, "p", "p", "p"]),
    "backproject_backward": lambda n, c, h, w, ho, wo: ("bbd_backproject_backward", [n, h, w, "p", "p", "p"]),
    "project_forward": lambda n, c, h, w, ho, wo: ("bbd_project_forward", [n, h, w, "p", "p", "eps", "p"]),
    "project_backward": lambda n, c, h, w, ho, wo: ("bbd_project_backward", [n, h, w, "p", "p", "eps", "p", "p", "p"]),
    "project_coords": lambda n, c, h, w, ho, wo: ("bbd_project_coords", [n, h, w, "p", "p", "p", "p", "p"]),
    "warp_forward": lambda n, c, h, w, ho, wo: ("bbd_warp_forward", [n, h, w, "p", "p", "p", "p", "p", "p"]),
    "pack_rgba": lambda n, c, h, w, ho, wo: ("bbd_pack_rgba", [n, h, w, "p", "p"]),
    "grid_sample_forward": lambda n, c, h, w, ho, wo: ("bbd_grid_sample_forward", [n, c, h, w, ho, wo, "p", "p", "p"]),
    "grid_sample_backward": lambda n, c, h, w, ho, wo: ("bbd_grid_sample_backward",
                                                        [n, c, h, w, ho, wo, "p", "p", "p", "p"]),
    "grid_sample_dest_keys": lambda n, c, h, w, ho, wo: ("bbd_grid_sample_dest_keys", [n, h, w, ho, wo, "p", "p"]),
    "grid_sample_backward_image": lambda n, c, h, w, ho, wo: ("bbd_grid_sample_backward_image",
                                                              [n, c, h, w, ho, wo, "p", "p", "p", "p", "p", "p"]),
    "ssim_forward": lambda n, c, h, w, ho, wo: ("bbd_ssim_forward", [n, c, h, w, "p", "p", "p"]),
    "ssim_backward": lambda n, c, h, w, ho, wo: ("bbd_ssim_backward", [n, c, h, w, "p", "p", "p", "p", "p"]),
    "pose_forward": lambda n, c, h, w, ho, wo: ("bbd_pose_forward", [n, "p", "p", 0, "p"]),
    "pose_backward": lambda n, c, h, w, ho, wo: ("bbd_pose_backward", [n, "p", "p", 0, "p", "p", "p"]),
    "pose_pack_forward": lambda n, c, h, w, ho, wo: ("bbd_pose_pack_forward", [n, "p", "p", "p", "p"]),
    "pose_pack_backward": lambda n, c, h, w, ho, wo: ("bbd_pose_pack_backward", [n, "p", "p", "p", "p"]),
}
HAS_IMAGE = [k for k in CALLS if not k.startswith("pose")]
HAS_CHANNELS = [k for k in CALLS if k.startswith(("grid_sample_forward", "grid_sample_backward", "ssim"))]
HAS_OUTPUT = [k for k in CALLS if k.startswith("grid_sample")]
GOOD = dict(n=2, c=3, h=8, w=8, ho=8, wo=8)


def _cases():
    out = []
    for k in CALLS:
        out.append((k, dict(GOOD, n=-1), E_ARG))
        out.append((k, dict(GOOD, n=0), 0))
    for k in HAS_IMAGE:
        out.append((k, dict(GOOD, h=-8), E_ARG))
        out.append((k, dict(GOOD, w=-8), E_ARG))
        out.append((k, dict(GOOD, n=1, h=65536, w=32768), E_RANGE))      # H*W = 2^31
    for k in HAS_CHANNELS:
        out.append((k, dict(GOOD, c=-3), E_ARG))
        out.append((k, dict(GOOD, n=65536, c=32768), E_RANGE))           # n*channels = 2^31
    for k in HAS_OUTPUT:
        out.append((k, dict(GOOD, ho=-8), E_ARG))
        out.append((k, dict(GOOD, wo=-8), E_ARG))
        out.append((k, dict(GOOD, n=1, ho=32768, wo=65536), E_RANGE))    # Ho*Wo = 2^31
    for k in ("ssim_forward", "ssim_backward"):
        out.append((k, dict(GOOD, h=1), E_RANGE))                       # reflection padding needs 2 rows
        out.append((k, dict(GOOD, w=1), E_RANGE))
    return out


CASES = _cases()


@pytest.mark.parametrize("call,sizes,want", CASES,
                         ids=[f"{k}-" + "-".join(f"{a}{v}" for a, v in s.items() if v != GOOD[a]) for k, s, _ in CASES])
def test_tier_a_sizes_are_checked_before_any_launch(lib_path, call, sizes, want):
    name, args = CALLS[call](**sizes)
    got = call_without_gpu(lib_path, name, args)
    assert got["rc"] == want, (name, sizes, got)
    if want == E_ARG:
        assert "negative" in got["msg"], got["msg"]


def test_project_chunks_of_unusable_sizes(lib_path):
    """The partial-sum count a caller allocates for bbd_project_backward: zero for sizes the call refuses."""
    import ctypes
    dll = ctypes.CDLL(lib_path)
    dll.bbd_project_chunks.restype = ctypes.c_int
    assert dll.bbd_project_chunks(192, 640) == 30
    assert dll.bbd_project_chunks(64, 64) == 1 and dll.bbd_project_chunks(17, 241) == 2
    assert dll.bbd_project_chunks(-8, 64) == 0 and dll.bbd_project_chunks(65536, 65536) == 0
