"""Tier B end to end: FusedLossMixin mixed into a trainer (kernels stepped on the CPU), against the losses,
gradients and warps the reference's own Trainer wrote into the golden cases.

The mixin replaces Trainer.generate_images_pred and Trainer.compute_losses; of the rest of the reference's
Trainer it reads the options and the sub-batch masks of valid_frames_trimin (trainer.py:888-981).  RecordedTrainer
carries exactly that, the masks from oracle.sub_batch_masks, which tests/test_oracle_golden.py pins to the masks
the reference recorded in every golden case.  On the GPU the same mixin is exercised through loss_step in
test_gpu_parity.py.
"""
import types

import pytest
import torch

from baseboostdepth_b200.trainer import FusedLossMixin
from fused_util import emu_backend
from helpers import Golden, rel_l2
from oracle import loss_path as O


class RecordedTrainer:
    """The state of the reference Trainer that FusedLossMixin reads."""

    def valid_frames_trimin(self, inputs):
        m = O.sub_batch_masks(inputs["ordering"], self.opt.frame_ids, self.valid_frames, self.opt.trimin)
        for attr, value in vars(m).items():
            setattr(self, attr, value)


class FusedTrainer(FusedLossMixin, RecordedTrainer):
    pass


@pytest.mark.parametrize("case", ["plain_mixed_s", "trimin_decomp"])
def test_reference_trainer_with_fused_mixin(case):
    g = Golden(case)
    tr = FusedTrainer.__new__(FusedTrainer)
    tr.opt = types.SimpleNamespace(**vars(g.opt()))
    tr.device, tr.num_scales, tr.maxing_valid_frames = torch.device("cpu"), g.num_scales, False
    tr._bbd_backend = emu_backend()
    tr.collect_ident = True
    tr.early_phase = 0                                  # a logging step: warps must be materialised
    tr.opt.frame_ids = O.frame_ids_from_ordering(g.ordering)
    tr.valid_frames = O.initial_valid_frames(g.ordering)
    tr.valid_frames_trimin(g.inputs)                    # the reference's own bookkeeping

    groups = [f for f in O.initial_valid_frames(g.ordering) if f == "s" or f > 0]
    raw = iter([g.noise[k] / 0.00001 for k in groups])   # the kernel applies the 1e-5 itself
    real_randn = torch.randn
    torch.randn = lambda *a, **k: next(raw)
    try:
        outputs = tr.generate_images_pred(g.inputs, g.outputs)
        losses = tr.compute_losses(g.inputs, outputs)
    finally:
        torch.randn = real_randn
    for k, v in g.losses.items():
        assert abs(float(losses[k]) - v) <= 2e-6, (k, float(losses[k]), v)
    losses["loss"].backward()
    for k, ref in g.grads.items():
        assert rel_l2(g.params[k].grad, ref) <= 1e-5, k
    s0 = g.scales[0]
    for k, ref in g.ref_out.items():
        if k[0] in ("color", "color_D") and k[2] == s0:
            assert (outputs[k] - ref).abs().max() <= 2e-5, k
        if k[0] == "depth":
            assert (outputs[k] - ref).abs().max() <= 1e-4, k
    if g.trimin:
        norm, guide = tr.ident
        assert any(len(v) for v in norm.values())


def test_incremental_pose_rows_are_masked_like_the_reference():
    """--incremental_skip (trainer.py:467-469): the pose stacks keep one row per row of the compacted frame
    stack and generate_images_pred masks them with valid_tri_mask[|f|].  The fused mixin must pick the same
    rows: on over-complete pose stacks its losses are the reference's golden losses of the compact stacks, the
    rows it picks get the gradients the oracle gives the compact stacks, and the other rows get none."""
    compact = Golden("trimin_mixed")
    poses = {k: v for k, v in compact.outputs.items() if k[0] == "cam_T_cam" and v.numel()}
    for v in poses.values():
        v.retain_grad()
    O.run(compact.inputs, compact.outputs, compact.opt(), compact.noise, num_scales=compact.num_scales)[0]["loss"].backward()

    g = Golden("trimin_mixed")
    tr = FusedTrainer.__new__(FusedTrainer)
    tr.opt = types.SimpleNamespace(**vars(g.opt()))
    tr.opt.incremental_skip = True
    tr.device, tr.num_scales, tr.maxing_valid_frames = torch.device("cpu"), g.num_scales, True
    tr._bbd_backend = emu_backend()
    tr.opt.frame_ids = O.frame_ids_from_ordering(g.ordering)
    tr.valid_frames = O.initial_valid_frames(g.ordering)
    tr.valid_frames_trimin(g.inputs)
    # over-complete pose stacks: the golden rows where the mask is set, other poses elsewhere
    gen = torch.Generator().manual_seed(77)
    leaves, masks = {}, {}
    for f in tr.valid_frames:
        if f == "s":
            continue
        masks[f] = torch.tensor(tr.valid_tri_mask[abs(f)])
        used = g.outputs[("cam_T_cam", 0, f)].detach()
        assert int(masks[f].sum()) == used.shape[0]
        full = torch.eye(4).repeat(len(masks[f]), 1, 1)
        full[:, :3, 3] = 0.05 * torch.randn(len(masks[f]), 3, generator=gen)
        full[masks[f]] = used
        leaves[f] = full.requires_grad_(True)
        g.outputs[("cam_T_cam", 0, f)] = leaves[f]
    groups = [f for f in O.initial_valid_frames(g.ordering) if f == "s" or f > 0]
    raw = iter([g.noise[k] / 0.00001 for k in groups])   # the kernel multiplies the raw draw by 1e-5 itself
    real_randn = torch.randn
    torch.randn = lambda *a, **k: next(raw)
    try:
        outputs = tr.generate_images_pred(g.inputs, g.outputs)
        losses = tr.compute_losses(g.inputs, outputs)
    finally:
        torch.randn = real_randn
    losses["loss"].backward()
    for k, v in g.losses.items():
        assert abs(float(losses[k]) - v) <= 2e-6, (k, float(losses[k]), v)
    for f, leaf in leaves.items():
        want = torch.zeros_like(leaf)
        want[masks[f]] = poses[("cam_T_cam", 0, f)].grad
        assert rel_l2(leaf.grad, want) <= 1e-5, f
