// TEST-ONLY host harness for the colour-frame gradients: the whole CPU harness of bbd_emu.cpp plus emu_* versions
// of bbd_frame_grad, bbd_frame_grad_stacks and bbd_smooth_image_grad, stepping the phase functions of
// baseboostdepth_b200/csrc/bbd_framegrad.cuh one pixel at a time.  Built into its own shared object
// (tests/frame_grad_util.py); never loaded by the package.  Exported symbols take HOST pointers.
#include "bbd_emu.cpp"
#include "../../baseboostdepth_b200/csrc/bbd_framegrad.cuh"

extern "C" {

int emu_frame_grad(const bbd_reproj_args* ap, const bbd_frame_grad_args* fp) {
  const bbd_reproj_args& a = *ap;
  const bbd_frame_grad_args& f = *fp;
  const int H = a.height, W = a.width;
  if (!a.no_ssim)
    for (int sb = 0; sb < a.num_scales * a.batch; ++sb)
      for (int q = 0; q < H * W; ++q) fg_coef_px(a, f, sb / a.batch, sb % a.batch, q / W, q % W);
  for (int b = 0; b < a.batch; ++b)
    for (int p = 0; p < H * W; ++p) fg_pred_px(a, f, b, p / W, p % W);
  return 0;
}

int emu_frame_grad_stacks(const bbd_reproj_args* ap, const bbd_frame_grad_args* fp) {
  const bbd_reproj_args& a = *ap;
  const bbd_frame_grad_args& f = *fp;
  const int HW = a.height * a.width, rows = fg_total_rows(f);
  if (!rows) return 0;
  const int n_items = a.num_scales * a.batch * a.max_rep * HW, n_keys = rows * HW;
  for (int i = 0; i <= n_items; ++i) gs_segment_mark(f.keys_sorted, n_items, n_keys, i, f.seg_start);
  for (int grow = 0; grow < rows; ++grow) {
    int slot, row;
    fg_locate_row(f, grow, slot, row);
    if (!f.gframes[slot]) continue;
    for (int c = 0; c < 3; ++c)
      for (int p = 0; p < HW; ++p) f.gframes[slot][((size_t)row * 3 + c) * HW + p] = fg_stack_px(a, f, slot, row, c, p);
  }
  return 0;
}

int emu_smooth_image_grad(const bbd_smooth_img_args* ap) {
  const bbd_smooth_img_args& a = *ap;
  for (int lvl = 0; lvl < a.levels; ++lvl) {
    if (!a.gimg[lvl]) continue;
    const int n = a.h[lvl] * a.w[lvl];
    for (int b = 0; b < a.batch; ++b)
      for (int i = 0; i < n; ++i) {
        float g[3];
        smi_px(a, lvl, b, i / a.w[lvl], i % a.w[lvl], g);
        for (int c = 0; c < 3; ++c) a.gimg[lvl][((size_t)b * 3 + c) * n + i] = g[c];
      }
  }
  return 0;
}

}  // extern "C"
