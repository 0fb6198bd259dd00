"""Every launch form of the loss kernels, as a table of production steps that reach it.

Each row is one step of ``trainer.loss_step``: a batch layout, a frame size and disparity pyramid, the switches
that select the form, and what the step must launch -- the fused-loss kernel (its exact template arguments, as
``bbd_reproj_kernel_name`` prints them), the identity pre-pass kernel, the disparity-backward kernels and whether
``reproj_finalize_kernel`` runs.  ``tests/test_launch_forms_gpu.py`` runs every row on the GPU against the oracle;
``tests/test_launch_emu.py`` checks that the rows name exactly the kernels the launch description
(``csrc/bbd_launch.cuh``) can produce.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple

# batch layouts: baselines per sample and the tri-minimisation flag (max_rep in the comment)
PM1 = dict(baselines=[1, 1], trimin=False)              # +-1: two candidates per sample
PM1_B1 = dict(baselines=[1], trimin=False)
STEREO = dict(baselines=["s", "s", "s"], trimin=False)  # one candidate per sample
TRI3 = dict(baselines=[1, "s", 1], trimin=True)         # three candidates at most: the tile form keeps them all
TRIMIN = dict(baselines=[3, 2, 1, "s"], trimin=True)    # one to six candidates: sweeps over candidate pairs

D2D_SINGLE = ("d2d_backward_fused_kernel",)
D2D_TWO_PASS = ("d2d_hpass_kernel", "d2d_backward_kernel")   # separable factors 2 / 4 / 8
D2D_GENERIC = ("d2d_backward_kernel",)                       # no separable level: no row pass


@dataclass(frozen=True)
class Case:
    name: str
    layout: Dict
    hw: Tuple[int, int]
    reproj: str                        # bbd_reproj_kernel_name of the step
    d2d: Tuple[str, ...] = D2D_SINGLE  # disparity backward kernels (grad steps)
    finalize: bool = False             # reproj_finalize_kernel runs
    scales: Tuple[int, ...] = (0, 1, 2, 3)
    factors: Optional[Tuple[int, ...]] = None   # disparity level s is (H/f_s, W/f_s); default 2**s
    grad: bool = True                  # False: the step runs under torch.no_grad()
    force_tile: bool = False           # fused._FORCE_TILE
    pipe: bool = False                 # BBD_PIPE=1
    split: bool = False                # fused._SPLIT_D2D_BACKWARD
    side: bool = True                  # fused._USE_SIDE
    no_winner: bool = False            # the backend withholds the winner plane (a C caller passing winner = NULL)
    offset_target: bool = False        # the target starts 4 bytes past a 16-byte boundary
    frame_grads: bool = False          # every colour frame requires grad
    seed: int = 11
    extra: Dict = field(default_factory=dict)

    @property
    def tile(self):
        return self.reproj.startswith("bbd::reproj_kernel<")

    @property
    def ident(self):
        return "ident_kernel" if self.tile else "ident_stream_kernel"

    @property
    def reproj_family(self):
        return self.reproj.split("::")[1].split("<")[0]


def _tma(k, g, m, wing=False):
    return f"bbd::reproj_stream_tma_kernel<{k}, {g}, {m}{', 1' if wing else ''}>"


def _plain(k, g, m, wing=False):
    return f"bbd::reproj_stream_kernel<{k}, {g}, {m}{', 1' if wing else ''}>"


PLAIN_HW = (50, 90)   # W = 2 (mod 4): no TMA, and the disparity backward takes the two-pass form

CASES = [
    # tile form ("exact mode"): every candidate kept resident up to three, reused from four
    Case("tile_keep_grad", PM1, (64, 96), "bbd::reproj_kernel<1, 1>", finalize=True, force_tile=True, frame_grads=True),
    Case("tile_keep_fwd", PM1, (64, 96), "bbd::reproj_kernel<0, 1>", finalize=True, force_tile=True, grad=False),
    Case("tile_keep3_grad", TRI3, (64, 96), "bbd::reproj_kernel<1, 1>", finalize=True, force_tile=True),
    Case("tile_reuse_grad", TRIMIN, (64, 96), "bbd::reproj_kernel<1, 0>", finalize=True, force_tile=True,
         frame_grads=True),
    Case("tile_reuse_fwd", TRIMIN, (64, 96), "bbd::reproj_kernel<0, 0>", finalize=True, force_tile=True, grad=False),
    # streaming form, TMA-staged planes
    Case("stream_k1_grad", STEREO, (48, 96), _tma(1, 1, 0), frame_grads=True),
    Case("stream_k1_fwd", STEREO, (48, 96), _tma(1, 0, 0), grad=False),
    Case("stream_k2_grad", PM1, (64, 96), _tma(2, 1, 0)),
    Case("stream_k2_fwd", PM1, (64, 96), _tma(2, 0, 0), grad=False),
    Case("multi_grad", TRIMIN, (64, 96), _tma(2, 1, 1, wing=True), finalize=True, frame_grads=True),
    Case("multi_fwd", TRIMIN, (64, 96), _tma(2, 0, 1), finalize=True, grad=False),
    Case("multi_grad_no_winner", TRIMIN, (64, 96), _tma(2, 1, 1), finalize=True, no_winner=True),
    # streaming form, plain loads because of the width
    Case("plain_k1_grad", STEREO, PLAIN_HW, _plain(1, 1, 0), D2D_TWO_PASS, scales=(0, 1), frame_grads=True),
    Case("plain_k1_fwd", STEREO, PLAIN_HW, _plain(1, 0, 0), scales=(0, 1), grad=False),
    Case("plain_k2_grad", PM1, PLAIN_HW, _plain(2, 1, 0), D2D_TWO_PASS, scales=(0, 1)),
    Case("plain_k2_fwd", PM1, PLAIN_HW, _plain(2, 0, 0), scales=(0, 1), grad=False),
    Case("plain_multi_grad", TRIMIN, PLAIN_HW, _plain(2, 1, 1, wing=True), D2D_TWO_PASS, finalize=True, scales=(0, 1)),
    Case("plain_multi_fwd", TRIMIN, PLAIN_HW, _plain(2, 0, 1), finalize=True, scales=(0, 1), grad=False),
    Case("plain_multi_grad_no_winner", TRIMIN, PLAIN_HW, _plain(2, 1, 1), D2D_TWO_PASS, finalize=True, scales=(0, 1),
         no_winner=True),
    # streaming form, plain loads because the target is not 16-byte aligned
    Case("plain_align_k2_grad", PM1, (64, 96), _plain(2, 1, 0), offset_target=True, frame_grads=True),
    Case("plain_align_multi_grad", TRIMIN, (64, 96), _plain(2, 1, 1, wing=True), finalize=True, offset_target=True),
    # pipelined form (opt-in)
    Case("pipe_k1_grad", STEREO, (64, 96), "bbd::reproj_pipe_kernel<1, 1>", pipe=True),
    Case("pipe_k1_fwd", STEREO, (64, 96), "bbd::reproj_pipe_kernel<1, 0>", pipe=True, grad=False),
    Case("pipe_k2_grad", PM1, (64, 96), "bbd::reproj_pipe_kernel<2, 1>", pipe=True),
    Case("pipe_k2_fwd", PM1, (64, 96), "bbd::reproj_pipe_kernel<2, 0>", pipe=True, grad=False),
    # disparity backward forms
    Case("d2d_generic_factors", PM1, (48, 96), _tma(2, 1, 0), D2D_GENERIC, scales=(0, 1, 2), factors=(1, 3, 6)),
    Case("d2d_wide_frame", PM1_B1, (16, 6152), _tma(2, 1, 0), D2D_TWO_PASS, scales=(0, 1)),
    Case("d2d_split", PM1, (64, 96), _tma(2, 1, 0), D2D_TWO_PASS, split=True),
    Case("no_side_streams", PM1, (64, 96), _tma(2, 1, 0), side=False),
    # segment rule at the edges: many short segments of a tall narrow frame, and tiny frames
    Case("tall_narrow", PM1, (260, 12), _tma(2, 1, 0), scales=(0, 1, 2)),
    Case("tiny_four_scales", PM1, (16, 16), _tma(2, 1, 0)),
]

BY_NAME = {c.name: c for c in CASES}
assert len(BY_NAME) == len(CASES)


def declared_kernel_names():
    return {c.reproj for c in CASES}
