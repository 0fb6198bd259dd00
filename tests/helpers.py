"""Shared test plumbing: golden-fixture loading and comparison metrics."""
from __future__ import annotations

import glob
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_cases():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def _parse_key(s):
    parts = s.split("|")
    if len(parts) == 1:
        return parts[0]
    out = []
    for p in parts:
        try:
            out.append(int(p))
        except ValueError:
            out.append(p)
    return tuple(out)


def _frame(s):
    return "s" if s == "s" else int(s)


class Golden:
    """One ``tests/golden/<case>.npz`` unpacked into trainer-style dicts."""

    def __init__(self, name, device="cpu", dtype=torch.float32):
        from baseboostdepth_b200.geometry import transformation_from_parameters
        from baseboostdepth_b200.synthetic import ordering_from_baselines

        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.name = name
        self.baselines = [_frame(m) for m in z["meta_baselines"]]
        self.scales = [int(s) for s in z["meta_scales"]]
        self.trimin, self.decomp, self.no_ssim = (bool(v) for v in z["meta_flags"])
        self.H, self.W = (int(v) for v in z["meta_hw"])
        self.num_scales = int(z["meta_num_scales"][0])
        self.valid_frames = [_frame(f) for f in z["meta_valid_frames"]]
        self.ordering = ordering_from_baselines(self.baselines)

        def T(a):
            return torch.from_numpy(np.asarray(a)).to(device=device, dtype=dtype)

        self.inputs = {"ordering": self.ordering}
        self.params, self.grads, self.noise, self.losses, self.ref_out, self.masks = {}, {}, {}, {}, {}, {}
        for k in z.files:
            kind, _, rest = k.partition(":")
            if kind == "in":
                self.inputs[_parse_key(rest)] = T(z[k])
            elif kind == "param":
                self.params[_parse_key(rest)] = T(z[k]).requires_grad_(True)
            elif kind == "grad":
                self.grads[_parse_key(rest)] = torch.from_numpy(z[k])
            elif kind == "noise":
                self.noise[_frame(rest)] = T(z[k])
            elif kind == "loss":
                self.losses[rest] = float(z[k])
            elif kind == "out":
                self.ref_out[_parse_key(rest)] = torch.from_numpy(z[k])
            elif kind == "mask":
                attr, _, key = rest.partition(":")
                self.masks.setdefault(attr, {})[key] = [bool(v) for v in z[k]]

        # rebuild outputs (disp, poses) from the leaf parameters exactly as synthetic.make_batch does
        self.outputs = {}
        for k, v in self.params.items():
            if k[0] == "disp":
                self.outputs[k] = v
        frames = sorted({k[1] for k in self.params if k[0] == "axisangle"}, key=lambda f: (abs(f), f < 0))
        for f in frames:
            Tm = transformation_from_parameters(self.params[("axisangle", f)], self.params[("translation", f)],
                                                invert=(f < 0))
            self.outputs[("cam_T_cam", 0, f)] = Tm
            if self.decomp:
                Te = Tm.clone().detach()
                Te[:, :3, 3:] /= 5.5
                self.outputs[("cam_T_cam_error", 0, f)] = Te
        top = max([m for m in self.baselines if m != "s"], default=0)
        for f in range(-top, top + 1):
            if f != 0 and ("cam_T_cam", 0, f) not in self.outputs:
                self.outputs[("cam_T_cam", 0, f)] = torch.zeros(0, 4, 4, device=device, dtype=dtype)
                if self.decomp:
                    self.outputs[("cam_T_cam_error", 0, f)] = torch.zeros(0, 4, 4, device=device, dtype=dtype)

    def opt(self):
        from oracle.loss_path import default_opt
        return default_opt(height=self.H, width=self.W, scales=list(self.scales), trimin=self.trimin,
                           decomp=self.decomp, no_ssim=self.no_ssim, pose_error=5.5,
                           batch_size=len(self.baselines))


def rel_l2(a, b):
    a = a.detach().double().cpu().reshape(-1)
    b = b.detach().double().cpu().reshape(-1)
    den = b.norm().item()
    return (a - b).norm().item() / den if den > 0 else (a - b).norm().item()


def max_abs(a, b):
    return (a.detach().double().cpu() - b.detach().double().cpu()).abs().max().item() if a.numel() else 0.0


# every gradient comparison of a test session lands here; tests/conftest.py writes it out at session end
PARITY_LOG = []


def assert_grad_parity(mine, ref32, ref64, key, tol=1e-5, case=None):
    """Gradient parity bar.

    Primary: relative L2 error against the fp32 oracle <= 1e-5 (BASELINE.md 5).  At full
    resolution the fp32 oracle itself sits 3e-3..9e-3 away from its own float64 evaluation:
    a single near-tie (argmin, |.| sign, border clip) that falls the other way moves an
    aggregated gradient by ~1/sqrt(N).  Where the primary bar is missed, the kernel must be
    no farther from the float64 evaluation than the fp32 oracle is (x2, + 2e-6).
    Which bar applied is recorded in PARITY_LOG (and printed when it is the secondary one).
    """
    e = rel_l2(mine, ref32)
    if ref64 is None:   # caller only has the float64 yardstick when the primary bar is missed
        assert e <= tol, (key, "vs fp32 oracle", e)
        PARITY_LOG.append({"case": case, "key": repr(key), "rel_l2_vs_fp32_oracle": e, "bar": "rel_l2_vs_fp32_oracle<=%g" % tol,
                           "passed": True})
        return e
    e_mine, e_ref = rel_l2(mine, ref64), rel_l2(ref32, ref64)
    bar = "rel_l2_vs_fp32_oracle<=%g" % tol if e <= tol else "no_farther_from_f64_than_fp32_oracle(x2+2e-6)"
    ok = e <= tol or e_mine <= 2.0 * e_ref + 2e-6
    PARITY_LOG.append({"case": case, "key": repr(key), "rel_l2_vs_fp32_oracle": e, "rel_l2_vs_f64": e_mine,
                       "fp32_oracle_vs_f64": e_ref, "bar": bar, "passed": bool(ok)})
    if e > tol:
        print(f"[parity] secondary bar for {case} {key}: vs fp32 oracle {e:.3e}, vs f64 {e_mine:.3e}, "
              f"oracle32 vs f64 {e_ref:.3e}")
    assert ok, (key, "vs fp32 oracle", e, "vs f64", e_mine, "oracle32 vs f64", e_ref)
    return e


def selection_check(win, plan, aux, scales, exact=False):
    """argmin planes equal the oracle's wherever its best-vs-runner-up margin exceeds 1e-6 (everywhere with
    ``exact``).  Returns the number of pixels that differ inside the margin."""
    order = [b for grp in aux["groups"] for b in plan.group_members[grp]]
    differ = 0
    for i, s in enumerate(scales):
        args = torch.cat(aux["argmin"][s], 0)
        mine = win[i].cpu()[order].long()
        agree = mine == args
        if bool(agree.all()):
            continue
        assert not exact, (s, int((~agree).sum()))
        margins = []
        for p in aux["planes"][s]:
            top = torch.topk(-p, 2, dim=1).values
            margins.append(top[:, 0] - top[:, 1])
        margin = torch.cat(margins, 0)
        assert bool((agree | (margin <= 1e-6)).all()), (s, int((~agree).sum()))
        differ += int((~agree).sum())
    return differ


def near_tie_mask(plan, aux, s, dilate=1):
    """(B,H,W) bool: pixels whose best-vs-runner-up margin in the oracle is <= 1e-6, dilated by `dilate`
    pixels (a selection that may legitimately differ changes the gradient of its 3x3 neighbourhood)."""
    import torch.nn.functional as F
    order = [b for grp in aux["groups"] for b in plan.group_members[grp]]
    margins = []
    for p in aux["planes"][s]:
        top = torch.topk(-p, 2, dim=1).values
        margins.append(top[:, 0] - top[:, 1])
    margin = torch.cat(margins, 0)
    near = torch.zeros_like(margin, dtype=torch.bool)
    near[order] = margin <= 1e-6
    if dilate:
        near = F.max_pool2d(near.float().unsqueeze(1), 2 * dilate + 1, 1, dilate)[:, 0] > 0
    return near


def pixel_agreement(mine, ref32, tol=1e-5):
    """Fraction of elements whose gradient differs by more than tol * max|ref|."""
    a, b = mine.detach().double().cpu(), ref32.detach().double().cpu()
    lim = tol * b.abs().max().item()
    return ((a - b).abs() > lim).double().mean().item()
