// Gradients of the fused view-synthesis loss with respect to the colour frames.
//
// The forward leaves the per-pixel winner of every scale in bbd_reproj_args.winner (index in candidate order:
// warped candidates, then identity candidates).  The reference differentiates only the winner's photometric
// term 0.85 mean_c SSIM(x, y) + 0.15 mean_c |y - x| at every target pixel; here that happens in three
// per-pixel gathers (no atomics, every sum in a fixed order):
//   1. fg_coef_px    per (scale, sample, centre q): SSIM window moments of the winner against the target and the
//                    coefficients (a, b, c) with d/dx(u) = a + b x(u) + c y(u), and the same for y(u), for the
//                    nine pixels u of the window around q (scaled by the upstream scalar of the scale);
//   2. fg_pred_px    per (sample, pixel p), all scales in order: d loss / d x_w(p) for every candidate w that
//                    wins somewhere in the 3x3 neighbourhood of p (reflection multiplicities, L1 at p itself),
//                    the target gradient and the identity-source gradients (both summed over scales), and for a
//                    warped candidate the plane g_pred plus the sort key (stack row, north-west tap) of p;
//   3. fg_stack_px   per stack pixel: the transpose of the bilinear border warp as a gather over the stably
//                    sorted keys (the scheme of gs_image_grad_px, extended to every scale, candidate and decomp
//                    twin that sampled the row; taps recomputed with project_pixel / make_taps, bit-identical
//                    to the forward), plus the identity-source gradients of the rows read unwarped.
// Entries of a candidate that wins nowhere in a pixel's neighbourhood get the key `n_keys` (sorted last, never
// gathered).  The smoothness image gradient (smi_px) is a separate per-pixel gather over the four edges of a
// pixel.  Same host/device phase structure as bbd_strip.cuh (tests/emu steps these functions on the CPU).
#pragma once
#include "bbd_common.cuh"

namespace bbd {

constexpr int FG_NCOEF = 6;  // per channel and window centre: x side (a, b, c), y side (a, b, c)

BBD_HD int fg_row_base(const bbd_frame_grad_args& f, int slot) {
  int base = 0;
  for (int i = 0; i < slot; ++i) base += f.stack_rows[i];
  return base;
}
BBD_HD int fg_total_rows(const bbd_frame_grad_args& f) { return fg_row_base(f, BBD_MAX_FRAMES); }

// source plane and (warped candidates) camera of candidate w of sample b; slot / row of its stack
BBD_HD const float* fg_source(const bbd_reproj_args& a, int b, int w, int n_rep, Cam& cam, int& slot, int& row) {
  const size_t img = (size_t)3 * a.height * a.width;
  if (w < n_rep) {
    const int32_t* e = a.tab.rep + ((size_t)b * BBD_MAX_REP + w) * 4;
    load_cam(cam, a.inv_K + (size_t)e[3] * 16, a.P + (size_t)e[2] * 12, a.width, a.height);
    slot = e[0]; row = e[1];
  } else {
    const int32_t* e = a.tab.ident + ((size_t)b * BBD_MAX_IDENT + (w - n_rep)) * 2;
    slot = e[0]; row = e[1];
  }
  return a.frames[slot] + (size_t)row * img;
}

// candidate value at pixel (px, py): the bilinear border warp (warped) or the pixel itself (identity)
BBD_HD void fg_value(const float* src, const Cam& cam, bool warped, float depth, int px, int py, int H, int W,
                     float x[3], int* nw_tap) {
  const int HW = H * W;
  if (!warped) {
    const int o = py * W + px;
    x[0] = src[o]; x[1] = src[HW + o]; x[2] = src[2 * HW + o];
    return;
  }
  Sample s;
  project_pixel(cam, px, py, depth, W, H, s);
  Taps t;
  make_taps(s, W, H, t);
  x[0] = tap_channel(src, t);
  x[1] = tap_channel(src + HW, t);
  x[2] = tap_channel(src + 2 * HW, t);
  if (nw_tap) *nw_tap = t.onw;
}

BBD_HD float fg_unit(const bbd_reproj_args& a) { return 1.0f / ((float)a.batch * (float)a.height * (float)a.width); }

// 1. SSIM coefficients of the winner's window around centre (qy, qx) of (scale s, sample b)
BBD_HD void fg_coef_px(const bbd_reproj_args& a, const bbd_frame_grad_args& f, int s, int b, int qy, int qx) {
  const int H = a.height, W = a.width, HW = H * W;
  const size_t sb = (size_t)s * a.batch + b;
  const int n_rep = a.tab.hdr[(size_t)b * 4];
  const int w = a.winner[sb * HW + (size_t)qy * W + qx];
  Cam cam;
  int slot, row;
  const float* src = fg_source(a, b, w, n_rep, cam, slot, row);
  const float* depth = a.depth + sb * HW;
  const float* tgt = a.target + (size_t)b * 3 * HW;
  float sx[3], sxx[3], sxy[3], sy[3], syy[3];
  bool first = true;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) {
      const int uy = reflect1(qy + dy, H), ux = reflect1(qx + dx, W), u = uy * W + ux;
      float x[3];
      fg_value(src, cam, w < n_rep, depth[u], ux, uy, H, W, x, nullptr);
      for (int c = 0; c < 3; ++c) {
        const float y = tgt[c * HW + u];
        if (first) { sx[c] = x[c]; sy[c] = y; sxx[c] = mul(x[c], x[c]); syy[c] = mul(y, y); sxy[c] = mul(x[c], y); }
        else {
          sx[c] = add(sx[c], x[c]); sy[c] = add(sy[c], y); sxx[c] = add(sxx[c], mul(x[c], x[c]));
          syy[c] = add(syy[c], mul(y, y)); sxy[c] = add(sxy[c], mul(x[c], y));
        }
      }
      first = false;
    }
  const float g = a.no_ssim ? 0.0f : f.gscale[s] * (fg_unit(a) * BBD_W_SSIM * BBD_THIRD);
  float* out = f.coef + sb * 3 * FG_NCOEF * HW + (size_t)qy * W + qx;
  for (int c = 0; c < 3; ++c) {
    WinX wx; wx.sx = sx[c]; wx.sxx = sxx[c]; wx.sxy = sxy[c];
    const WinY wy = target_stats(sy[c], syy[c]);
    SsimParts q;
    ssim_channel(wx, wy, q);
    float k[FG_NCOEF];
    ssim_coefs(q, wy, g, k[0], k[1], k[2]);
    ssim_coefs_y(q, wy, g, k[3], k[4], k[5]);
    for (int i = 0; i < FG_NCOEF; ++i) out[(size_t)(c * FG_NCOEF + i) * HW] = k[i];
  }
}

// 2. d loss / d x_w(p) of the candidates winning around pixel (py, px) of sample b, all scales
BBD_HD void fg_pred_px(const bbd_reproj_args& a, const bbd_frame_grad_args& f, int b, int py, int px) {
  const int H = a.height, W = a.width, HW = H * W, p = py * W + px;
  const int n_rep = a.tab.hdr[(size_t)b * 4], n_id = a.tab.hdr[(size_t)b * 4 + 1];
  const int n_keys = fg_total_rows(f) * HW;
  const float* tgt = a.target + (size_t)b * 3 * HW;
  const float y[3] = {tgt[p], tgt[HW + p], tgt[2 * HW + p]};
  const float g_l1_unit = a.no_ssim ? fg_unit(a) * BBD_THIRD : fg_unit(a) * BBD_W_L1 * BBD_THIRD;
  float gt[3] = {0.0f, 0.0f, 0.0f};
  float gid[BBD_MAX_IDENT][3];
  for (int j = 0; j < BBD_MAX_IDENT; ++j) gid[j][0] = gid[j][1] = gid[j][2] = 0.0f;
  for (int s = 0; s < a.num_scales; ++s) {
    const size_t sb = (size_t)s * a.batch + b;
    const uint8_t* win = a.winner + sb * HW;
    const float* cf = a.no_ssim ? nullptr : f.coef + sb * 3 * FG_NCOEF * HW;
    const float g_l1 = f.gscale[s] * g_l1_unit;
    // window centres whose window holds p, with the multiplicity of p in it (a reflected border pixel sits twice)
    int wq[9], oq[9];
    float mq[9];
    int nq = 0;
    if (a.no_ssim) {
      wq[0] = win[p]; oq[0] = p; mq[0] = 1.0f; nq = 1;
    } else {
      for (int dy = -1; dy <= 1; ++dy) {
        const int cy = py + dy;
        if (cy < 0 || cy >= H) continue;
        const float my = ((py == 1 && dy == -1) || (py == H - 2 && dy == 1)) ? 2.0f : 1.0f;
        for (int dx = -1; dx <= 1; ++dx) {
          const int cx = px + dx;
          if (cx < 0 || cx >= W) continue;
          const float m = my * (((px == 1 && dx == -1) || (px == W - 2 && dx == 1)) ? 2.0f : 1.0f);
          wq[nq] = win[cy * W + cx]; oq[nq] = cy * W + cx; mq[nq] = m; ++nq;
        }
      }
    }
    const int own = win[p];
    unsigned written = 0u;
    for (int i = 0; i < nq; ++i) {
      const int w = wq[i];
      bool seen = false;
      for (int j = 0; j < i; ++j) seen = seen || wq[j] == w;
      if (seen) continue;
      Cam cam;
      int slot, row, tap = 0;
      const bool warped = w < n_rep;
      const float* src = fg_source(a, b, w, n_rep, cam, slot, row);
      float x[3];
      fg_value(src, cam, warped, a.depth[sb * HW + p], px, py, H, W, x, &tap);
      float gx[3] = {0.0f, 0.0f, 0.0f};
      if (cf)
        for (int j = i; j < nq; ++j) {
          if (wq[j] != w) continue;
          for (int c = 0; c < 3; ++c) {
            const float* k = cf + (size_t)(c * FG_NCOEF) * HW + oq[j];
            gx[c] += mq[j] * (k[0] + k[(size_t)HW] * x[c] + k[(size_t)2 * HW] * y[c]);
            gt[c] += mq[j] * (k[(size_t)3 * HW] + k[(size_t)4 * HW] * y[c] + k[(size_t)5 * HW] * x[c]);
          }
        }
      if (own == w)
        for (int c = 0; c < 3; ++c) {
          const float d = sub(y[c], x[c]);  // l1 = |target - pred|; abs'(0) = 0
          const float sg = (d > 0.0f) ? g_l1 : ((d < 0.0f) ? -g_l1 : 0.0f);
          gx[c] -= sg;
          gt[c] += sg;
        }
      if (warped) {
        written |= 1u << w;
        float* gp = f.gpred + (sb * a.max_rep + w) * 3 * HW + p;
        gp[0] = gx[0]; gp[HW] = gx[1]; gp[2 * HW] = gx[2];
        f.keys[(sb * a.max_rep + w) * HW + p] = (fg_row_base(f, slot) + row) * HW + tap;
      } else {
        for (int c = 0; c < 3; ++c) gid[w - n_rep][c] += gx[c];
      }
    }
    for (int k = 0; k < a.max_rep; ++k)
      if (!(written & (1u << k))) f.keys[(sb * a.max_rep + k) * HW + p] = n_keys;
  }
  if (f.gtarget)
    for (int c = 0; c < 3; ++c) f.gtarget[((size_t)b * 3 + c) * HW + p] = gt[c];
  for (int j = 0; j < n_id; ++j)
    for (int c = 0; c < 3; ++c) f.gident[(((size_t)b * BBD_MAX_IDENT + j) * 3 + c) * HW + p] = gid[j][c];
}

// 3. gradient of stack row `grow` (rows of all stacks counted in slot order), channel c, pixel p
BBD_HD float fg_stack_px(const bbd_reproj_args& a, const bbd_frame_grad_args& f, int slot, int row, int c, int p) {
  const int H = a.height, W = a.width, HW = H * W;
  const int y = p / W, x = p - y * W;
  const int base = (fg_row_base(f, slot) + row) * HW;
  float acc = 0.0f;
  // role r: this pixel is the (NW, NE, SW, SE) tap of the entries whose north-west tap is (p, p-1, p-W, p-W-1)
  for (int r = 0; r < 4; ++r) {
    const int dx = r & 1, dy = r >> 1;
    if ((dx && x == 0) || (dy && y == 0)) continue;
    const int key = base + p - dx - dy * W;
    for (int i = f.seg_start[key]; i < f.seg_start[key + 1]; ++i) {
      const int e = f.order[i];  // ((s * B + b) * max_rep + k) * HW + q
      const int q = e % HW, sbk = e / HW, k = sbk % a.max_rep, sb = sbk / a.max_rep, b = sb % a.batch;
      const int32_t* t = a.tab.rep + ((size_t)b * BBD_MAX_REP + k) * 4;
      Cam cam;
      load_cam(cam, a.inv_K + (size_t)t[3] * 16, a.P + (size_t)t[2] * 12, W, H);
      Sample smp;
      project_pixel(cam, q % W, q / W, a.depth[(size_t)sb * HW + q], W, H, smp);
      Taps tp;
      make_taps(smp, W, H, tp);
      const float wt = (r == 0) ? tp.wnw : ((r == 1) ? tp.wne : ((r == 2) ? tp.wsw : tp.wse));
      acc = fma_(f.gpred[((size_t)sbk * 3 + c) * HW + q], wt, acc);
    }
  }
  // identity candidates read the row unwarped
  for (int b = 0; b < a.batch; ++b) {
    const int n_id = a.tab.hdr[(size_t)b * 4 + 1];
    for (int j = 0; j < n_id; ++j) {
      const int32_t* e = a.tab.ident + ((size_t)b * BBD_MAX_IDENT + j) * 2;
      if (e[0] == slot && e[1] == row) acc = add(acc, f.gident[(((size_t)b * BBD_MAX_IDENT + j) * 3 + c) * HW + p]);
    }
  }
  return acc;
}

// slot and row of global stack row `grow`
BBD_HD void fg_locate_row(const bbd_frame_grad_args& f, int grow, int& slot, int& row) {
  slot = 0;
  while (slot < BBD_MAX_FRAMES - 1 && grow >= f.stack_rows[slot]) { grow -= f.stack_rows[slot]; ++slot; }
  row = grow;
}

// ---- smoothness: gradient w.r.t. the colour level ------------------------------------------------------------
// L = mean_x |dx d| e^{-mean_c |dx I|} + mean_y (same), d = r * disp (r = 1/(mean+1e-7) or 1).  Pixel (y, x) of
// channel c is an end of at most four edges; edge e with I-difference D_c = I_c(first) - I_c(second) contributes
//   -/+ r |dd_e| e^{-mean_c|D|} sign(D_c) / (3 N)       (- for the first pixel of the edge, + for the second).
BBD_HD void smi_px(const bbd_smooth_img_args& a, int lvl, int b, int y, int x, float g[3]) {
  const int h = a.h[lvl], w = a.w[lvl], n = h * w;
  const float* d = a.disp[lvl] + (size_t)b * n;
  const float* img = a.img[lvl] + (size_t)b * 3 * n;
  const float r = a.coef ? a.coef[((size_t)lvl * a.batch + b) * 2] : 1.0f;
  const float inx = 1.0f / ((float)a.batch * (float)h * (float)(w - 1));
  const float iny = 1.0f / ((float)a.batch * (float)(h - 1) * (float)w);
  g[0] = g[1] = g[2] = 0.0f;
  // (first pixel, second pixel, this pixel's sign, normaliser) of the four edges
  const int o = y * w + x;
  const int firsts[4] = {o, o - 1, o, o - w};
  const int seconds[4] = {o + 1, o, o + w, o};
  const bool have[4] = {x + 1 < w, x > 0, y + 1 < h, y > 0};
  const float side[4] = {-1.0f, 1.0f, -1.0f, 1.0f};
  for (int e = 0; e < 4; ++e) {
    if (!have[e]) continue;
    const int i0 = firsts[e], i1 = seconds[e];
    float D[3], s = 0.0f;
    for (int c = 0; c < 3; ++c) {
      D[c] = img[c * n + i0] - img[c * n + i1];
      s += fabsf(D[c]);
    }
    const float k = side[e] * r * fabsf(d[i0] - d[i1]) * expf(-s * BBD_THIRD) * BBD_THIRD * (e < 2 ? inx : iny);
    for (int c = 0; c < 3; ++c) g[c] += (D[c] > 0.0f) ? k : ((D[c] < 0.0f) ? -k : 0.0f);
  }
  const float sc = a.gscale[lvl];
  for (int c = 0; c < 3; ++c) g[c] *= sc;
}

}  // namespace bbd
