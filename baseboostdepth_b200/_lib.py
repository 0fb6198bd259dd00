"""ctypes binding of ``libbbd_loss.so`` (C ABI in ``include/bbd_loss.h``).

The library is built in-tree by ``baseboostdepth_b200/build.py`` (``nvcc`` for
sm_100a).  There is no CPU implementation: if the shared object is missing or
a tensor is not on a CUDA device the call raises.  (``tests/emu`` builds a
host harness that steps the same kernel source on the CPU; tests inject it
through the ``backend=`` argument of the ops, the package never loads it.)
"""
from __future__ import annotations

import ctypes as C
import os

import torch

MAX_FRAMES, MAX_GROUPS, MAX_REP, MAX_IDENT, MAX_SCALES = 16, 8, 12, 6, 4
LIB_NAME = "libbbd_loss.so"
LIB_PATH = os.environ.get("BBD_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

fp = C.c_void_p


class Tables(C.Structure):
    _fields_ = [("hdr", fp), ("rep", fp), ("ident", fp)]


class IdentArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("no_ssim", C.c_int32),
                ("target", fp), ("frames", fp * MAX_FRAMES), ("noise", fp * MAX_GROUPS),
                ("noise_scale", C.c_float), ("tab", Tables), ("ident_min", fp), ("ident_arg", fp),
                ("frames_rgba", fp * MAX_FRAMES), ("force_tile", C.c_int32)]


class ReprojArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("num_scales", C.c_int32),
                ("no_ssim", C.c_int32), ("need_grad", C.c_int32), ("max_rep", C.c_int32), ("num_pose", C.c_int32),
                ("target", fp), ("frames", fp * MAX_FRAMES), ("depth", fp), ("inv_K", fp), ("P", fp),
                ("ident_min", fp), ("tab", Tables), ("loss_part", fp), ("gpose_part", fp), ("gdepth", fp),
                ("winner", fp), ("ident_arg", fp), ("frames_rgba", fp * MAX_FRAMES), ("min_rep", C.c_int32),
                ("tickets", fp), ("pair_sum", fp), ("loss_out", fp), ("gpose_out", fp), ("force_tile", C.c_int32)]


class SmoothArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("levels", C.c_int32), ("h", C.c_int32 * MAX_SCALES),
                ("w", C.c_int32 * MAX_SCALES), ("disp", fp * MAX_SCALES), ("img", fp * MAX_SCALES),
                ("gdisp", fp * MAX_SCALES), ("scratch", fp), ("loss", fp), ("max_chunks", C.c_int32),
                ("normalize", C.c_int32), ("defer_norm", C.c_int32), ("coef", fp)]


class D2DArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("levels", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
                ("h", C.c_int32 * MAX_SCALES), ("w", C.c_int32 * MAX_SCALES), ("min_disp", C.c_float),
                ("disp_span", C.c_float), ("sql", C.c_int32), ("disp", fp * MAX_SCALES), ("depth", fp),
                ("gdepth", fp), ("gscale", fp), ("gsmooth", fp * MAX_SCALES), ("gsmooth_scale", fp), ("gsmooth_coef", fp),
                ("gdisp", fp * MAX_SCALES), ("scratch", fp)]


class FrameGradArgs(C.Structure):
    _fields_ = [("gscale", fp), ("stack_rows", C.c_int32 * MAX_FRAMES), ("coef", fp), ("gpred", fp), ("keys", fp),
                ("gident", fp), ("gtarget", fp), ("keys_sorted", fp), ("order", fp), ("seg_start", fp),
                ("gframes", fp * MAX_FRAMES)]


class SmoothImgArgs(C.Structure):
    _fields_ = [("batch", C.c_int32), ("levels", C.c_int32), ("h", C.c_int32 * MAX_SCALES),
                ("w", C.c_int32 * MAX_SCALES), ("disp", fp * MAX_SCALES), ("img", fp * MAX_SCALES), ("coef", fp),
                ("gscale", fp), ("gimg", fp * MAX_SCALES)]


# every symbol include/bbd_loss.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "bbd_version", "bbd_last_error_string", "bbd_reproj_tiles", "bbd_ident_forward", "bbd_reproj_fused",
    "bbd_reproj_finalize", "bbd_warp_forward", "bbd_smooth_scratch_floats", "bbd_smooth_fused",
    "bbd_disp_to_depth_forward", "bbd_disp_to_depth_backward", "bbd_disp_to_depth_backward_pass1",
    "bbd_disp_to_depth_backward_pass2", "bbd_d2d_scratch_floats", "bbd_backproject_forward",
    "bbd_backproject_backward", "bbd_project_forward", "bbd_project_chunks", "bbd_project_backward",
    "bbd_ssim_forward", "bbd_ssim_backward", "bbd_pose_pack_forward", "bbd_pose_pack_backward",
    "bbd_pose_forward", "bbd_pose_backward", "bbd_grid_sample_forward", "bbd_grid_sample_backward",
    "bbd_grid_sample_dest_keys", "bbd_grid_sample_backward_image",
    "bbd_u8_to_f32", "bbd_loss_combine_forward", "bbd_loss_combine_backward", "bbd_pack_rgba", "bbd_project_coords", "bbd_reproj_kernel_name", "bbd_reproj_finalizes_itself",
    "bbd_frame_grad", "bbd_frame_grad_stacks", "bbd_smooth_image_grad",
]


def ptr(t):
    """Device (or, for the emulator, host) address of a contiguous tensor; None -> NULL."""
    if t is None:
        return None
    assert t.is_contiguous(), "bbd: tensor must be contiguous"
    return t.data_ptr()


class Backend:
    """A loaded shared object plus its calling convention (symbol prefix, stream argument)."""

    def __init__(self, path, prefix="bbd_", cuda=True):
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found: build it with `python -m baseboostdepth_b200.build` "
                f"(nvcc, sm_100a). There is no fallback implementation.")
        self.dll = C.CDLL(path)
        self.prefix = prefix
        self.cuda = cuda
        self.path = path
        self.launches = 0   # kernels enqueued through this binding (bench.py reports it)
        for name in ("reproj_tiles", "project_chunks"):
            getattr(self.dll, prefix + name).restype = C.c_int
        getattr(self.dll, prefix + "smooth_scratch_floats").restype = C.c_size_t
        getattr(self.dll, prefix + "d2d_scratch_floats").restype = C.c_size_t
        if cuda:
            self.dll.bbd_last_error_string.restype = C.c_char_p
            self.dll.bbd_reproj_kernel_name.restype = C.c_char_p

    def check_device(self, *tensors):
        dev = None
        for t in tensors:
            if t is None:
                continue
            if self.cuda and not t.is_cuda:
                raise RuntimeError("bbd: tensors must live on a CUDA device (there is no CPU path)")
            if self.cuda:
                # kernels are launched on torch's current device / stream with raw pointers: every tensor has
                # to live there (one process drives one GPU; set it with torch.cuda.set_device)
                if dev is None:
                    dev = t.device
                    if dev.index is not None and dev.index != torch.cuda.current_device():
                        raise RuntimeError(f"bbd: tensors live on {dev} but the current CUDA device is "
                                           f"cuda:{torch.cuda.current_device()} (call torch.cuda.set_device first)")
                elif t.device != dev:
                    raise RuntimeError(f"bbd: tensors on different devices ({dev} and {t.device})")
            if t.dtype not in (torch.float32, torch.int32, torch.uint8):
                raise RuntimeError(f"bbd: unsupported dtype {t.dtype} (the path is fp32 only)")

    def stream(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(self, name, *args):
        fn = getattr(self.dll, self.prefix + name)
        if self.cuda:
            args = args + (self.stream(),)
        rc = fn(*args)
        self.launches += {"grid_sample_backward_image": 2, "frame_grad": 2, "frame_grad_stacks": 2}.get(name, 1)
        if rc != 0:
            msg = self.dll.bbd_last_error_string().decode() if self.cuda else ""
            raise RuntimeError(f"bbd_{name} failed with code {rc}: {msg}")

    def value(self, name, *args):
        return getattr(self.dll, self.prefix + name)(*args)


_CUDA = None


def cuda_backend() -> Backend:
    global _CUDA
    if _CUDA is None:
        if not torch.cuda.is_available():
            raise RuntimeError("bbd: no CUDA device; the view-synthesis loss has no CPU implementation")
        _CUDA = Backend(LIB_PATH, "bbd_", cuda=True)
        if _CUDA.dll.bbd_version() != 2:
            raise RuntimeError("bbd: ABI version mismatch; rebuild libbbd_loss.so")
    return _CUDA
