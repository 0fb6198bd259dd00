// TEST-ONLY host harness: steps the thread-block phases of the sm_100a kernels on the CPU.
//
// The device kernels in baseboostdepth_b200/csrc/bbd_kernels.cu are thin drivers around the
// __host__ __device__ phase functions of bbd_strip.cuh / bbd_stream.cuh / bbd_pipe.cuh /
// bbd_smooth.cuh / bbd_ops.cuh / bbd_framegrad.cuh.  This file instantiates the same phase
// functions with g++ and steps the launches bbd_launch.cuh describes: for every block, each
// phase for tid = 0..NT-1 before moving to the next (a barrier between phases), so index
// logic, halo/reflection handling, candidate tables and the analytic gradients can be
// checked against the oracle in the GPU-less build container.  It is never loaded by the
// package; exported symbols are emu_* and take HOST pointers.
#include <stdlib.h>
#include <string.h>

#include <vector>

#define BBD_EMU 1
#include "simt.h"
#include "../../baseboostdepth_b200/csrc/bbd_launch.cuh"
#include "../../baseboostdepth_b200/csrc/bbd_pipe.cuh"
#include "../../baseboostdepth_b200/csrc/bbd_framegrad.cuh"

using namespace bbd;
#define FOR_STID for (int tid = 0; tid < SCfg::NT; ++tid)

// The launch decisions (bbd_launch.cuh) are taken for a B200: 148 SMs and a tensor-map encoder
// (-DBBD_EMU_NO_TMA steps the plain-load kernels instead).
static LaunchDevice b200() {
#ifdef BBD_EMU_NO_TMA
  return {148, false, pipe_requested()};
#else
  return {148, true, pipe_requested()};
#endif
}

extern "C" {

// number of significands (all 2^23, three binades) for which div_const(a, d, RN(1/d)) != a / d
long emu_div_const_mismatches(float d) {
  const float y = 1.0f / d;
  long bad = 0;
  const uint32_t exps[3] = {100u, 127u, 140u};
  for (int e = 0; e < 3; ++e)
    for (uint32_t m = 0; m < (1u << 23); ++m) {
      const uint32_t bits = (exps[e] << 23) | m;
      float a;
      memcpy(&a, &bits, 4);
      if (div_const(a, d, y) != a / d) ++bad;
    }
  return bad;
}

int emu_reproj_tiles(int32_t height, int32_t width) { return reproj_slots(height, width); }

int emu_project_coords(int32_t n, int32_t H, int32_t W, const float* depth, const float* inv_K, const float* P, float* grid,
                       float* pix) {
  for (int b = 0; b < n; ++b)
    for (int i = 0; i < H * W; ++i) stream_coords_px(H, W, depth, inv_K, P, b, i / W, i % W, grid, pix);
  return 0;
}

long emu_skipped_sweeps_total(void) { return emu_skipped_sweeps(); }

int emu_pack_rgba(int32_t n, int32_t H, int32_t W, const float* planar, float* rgba) {
  const size_t HW = (size_t)H * W;
  for (size_t img = 0; img < (size_t)n; ++img)
    for (size_t j = 0; j < HW; ++j) {
      float* o = rgba + (img * HW + j) * 4;
      o[0] = planar[img * 3 * HW + j];
      o[1] = planar[img * 3 * HW + HW + j];
      o[2] = planar[img * 3 * HW + 2 * HW + j];
      o[3] = 0.0f;
    }
  return 0;
}

}  // extern "C"
// one launch of the streaming or pipelined form: every unit (warp, or block of the pipelined form) in turn
template <int K, bool GRAD, bool MULTI, bool WING>
static void emu_stream(const bbd_reproj_args& a, const ReprojLaunch& L, const KernelLaunch& l) {
  std::vector<float> smem(StreamSmem<K, true, MULTI>::FLOATS + StreamSmem<K, false, MULTI>::FLOATS + PipeSmem<K, GRAD>::FLOATS);
  StreamTmaMaps none = {nullptr, nullptr, nullptr};
  for (int unit = 0; unit < l.units; ++unit) {
    if (L.form == REPROJ_PIPE)
      simt::run_block(GRAD ? 96 : 64, [&](int tid) { pipe_unit<K, GRAD>(a, unit, tid, smem.data(), L.stride, none, l.seg_rows); });
    else if (L.tma)
      simt::run_block(32, [&](int tid) { stream_unit<K, GRAD, true, MULTI, WING>(a, unit, tid, smem.data(), L.stride, none, l.seg_rows); });
    else
      simt::run_block(32, [&](int tid) { stream_unit<K, GRAD, false, MULTI, WING>(a, unit, tid, smem.data(), L.stride, none, l.seg_rows); });
  }
}
extern "C" {

int emu_ident_forward(const bbd_ident_args* ap) {
  const bbd_ident_args& a = *ap;
  if (!rgba_aligned(a.frames_rgba)) return BBD_E_ARG;
  const IdentLaunch L = ident_launch(a, b200().sms);
  if (L.stream) {
    for (int unit = 0; unit < L.units; ++unit)
      simt::run_block(32, [&](int tid) { ident_unit(a, const_cast<float* const*>(a.frames_rgba), unit, tid, L.seg_rows); });
    return 0;
  }
  std::vector<float> smem(IdentStripSmem<SCfg>::floats());
  std::vector<StripCtx> ctx(SCfg::NT);
  const int H = a.height, W = a.width;
  const int gx = (W + SCfg::TW - 1) / SCfg::TW, gy = (H + SCfg::TH - 1) / SCfg::TH;
  for (int bz = 0; bz < a.batch; ++bz)
    for (int by = 0; by < gy; ++by)
      for (int bx = 0; bx < gx; ++bx) {
        IdentStripSmem<SCfg> sm;
        sm.carve(smem.data());
        FOR_STID ctx[tid] = make_strip<SCfg>(bx, by, bz, tid, a.batch, H, W);
        const int b = ctx[0].b;
        const int32_t* hdr = a.tab.hdr + (size_t)b * 4;
        const int n_id = hdr[1];
        const float* noise = a.noise[hdr[2]] + (size_t)hdr[3] * H * W;
        FOR_STID is_load<SCfg>(a.target + (size_t)b * 3 * H * W, sm.tgt, ctx[tid], H, W);
        FOR_STID is_target_stats<SCfg>(a, sm, ctx[tid]);
        for (int j = 0; j < n_id; ++j) {
          const int32_t* e = a.tab.ident + ((size_t)b * BBD_MAX_IDENT + j) * 2;
          FOR_STID is_load<SCfg>(a.frames[e[0]] + (size_t)e[1] * 3 * H * W, sm.src, ctx[tid], H, W);
          FOR_STID is_candidate<SCfg>(a, sm, ctx[tid], j, noise);
        }
        FOR_STID is_store<SCfg>(a, sm, ctx[tid]);
      }
  return 0;
}

int emu_reproj_fused(const bbd_reproj_args* ap) {
  const bbd_reproj_args& a = *ap;
  if (!rgba_aligned(a.frames_rgba)) return BBD_E_ARG;
  const ReprojLaunch L = reproj_launch(a, b200());
  if (L.form != REPROJ_TILE) {
    for (int i = 0; i < L.n_launches; ++i)
      with_stream_instance(L, L.launch[i], [&](auto k, auto grad, auto multi, auto wing) {
        emu_stream<decltype(k)::value, decltype(grad)::value, decltype(multi)::value, decltype(wing)::value>(a, L, L.launch[i]);
      });
    return 0;
  }
  const bool keep = L.keep;
  std::vector<float> smem(L.tile_smem / sizeof(float));
  std::vector<float> red(12 * SCfg::NT + 12 * SCfg::RED_SEG * 2);  // host-side reduction scratch
  std::vector<float> gPs((size_t)SCfg::NT * 12), parts(SCfg::NT);
  std::vector<StripCtx> ctx(SCfg::NT);
  const int gx = (a.width + SCfg::TW - 1) / SCfg::TW, gy = (a.height + SCfg::TH - 1) / SCfg::TH;
  for (int bz = 0; bz < a.num_scales * a.batch; ++bz)
    for (int by = 0; by < gy; ++by)
      for (int bx = 0; bx < gx; ++bx) {
        StripSmem<SCfg> sm;
        sm.carve(smem.data(), keep ? a.max_rep : 1);
        sm.red = red.data();
        FOR_STID ctx[tid] = make_strip<SCfg>(bx, by, bz, tid, a.batch, a.height, a.width);
        const int b = ctx[0].b, tile = ctx[0].tile, ntiles = ctx[0].ntiles;
        const int n_rep = a.tab.hdr[(size_t)b * 4];
        FOR_STID rs_load_target<SCfg>(a, sm, ctx[tid], tid);
        FOR_STID rs_target_stats<SCfg>(a, sm, ctx[tid]);
        {
          const int s = ctx[0].s;
          FOR_STID rs_begin_scale<SCfg>(sm, tid);
          for (int k = 0; k < n_rep; ++k) {
            if (keep) {
              FOR_STID rs_warp<SCfg, true>(a, sm, ctx[tid], k);
              FOR_STID rs_stats<SCfg, true>(a, sm, ctx[tid], k);
            } else {
              FOR_STID rs_warp<SCfg, false>(a, sm, ctx[tid], k);
              FOR_STID rs_stats<SCfg, false>(a, sm, ctx[tid], k);
            }
          }
          FOR_STID parts[tid] = rs_select<SCfg>(a, sm, ctx[tid], n_rep);
          FOR_STID rs_park<SCfg, 1>(sm.red, tid, &parts[tid]);
          FOR_STID rs_level1<SCfg, 1>(sm.red, tid);
          FOR_STID rs_level2<SCfg, 1>(sm.red, tid, a.loss_part + ((size_t)s * a.batch + b) * ntiles + tile);
          if (!a.need_grad) continue;
          for (int k = 0; k < BBD_MAX_REP; ++k) {
            float* out = a.gpose_part + ((((size_t)s * a.batch + b) * BBD_MAX_REP + k) * ntiles + tile) * 12;
            if (k >= n_rep || !sm.anywin[k]) {
              for (int i = 0; i < 12; ++i) out[i] = 0.0f;
              continue;
            }
            {
              const float* src;
              Cam cam;
              rs_candidate(a, b, k, src, cam);
              for (size_t i = 0; i < gPs.size(); ++i) gPs[i] = 0.0f;
              for (int m = 0; m * SCfg::NW < SCfg::TH; m += BBD_BWD_ROWS) {   // BBD_BWD_ROWS rows per warp at a time, lanes in lockstep
                for (int r = 0; r < BBD_BWD_ROWS; ++r)
                  FOR_STID { const int q = ctx[tid].warp + (m + r) * SCfg::NW; if (q < SCfg::TH) rs_bwd_vertical<SCfg>(a, sm, ctx[tid], k, q, r); }
                for (int r = 0; r < BBD_BWD_ROWS; ++r)
                  FOR_STID { const int q = ctx[tid].warp + (m + r) * SCfg::NW; if (q < SCfg::TH) { if (keep) rs_bwd_horizontal<SCfg, true>(a, sm, ctx[tid], k, q, src, cam, &gPs[(size_t)tid * 12], r); else rs_bwd_horizontal<SCfg, false>(a, sm, ctx[tid], k, q, src, cam, &gPs[(size_t)tid * 12], r); } }
              }
            }
            FOR_STID rs_park<SCfg, 12>(sm.red, tid, &gPs[(size_t)tid * 12]);
            FOR_STID rs_level1<SCfg, 12>(sm.red, tid);
            FOR_STID rs_level2<SCfg, 12>(sm.red, tid, out);
          }
          FOR_STID rs_store_gdepth<SCfg>(a, sm, ctx[tid]);
        }
      }
  return 0;
}

const char* emu_reproj_kernel_name(const bbd_reproj_args* a) {
  if (!a) return "";
  static char name[64];
  reproj_kernel_name(reproj_launch(*a, b200()), name, sizeof(name));
  return name;
}
int emu_reproj_finalizes_itself(const bbd_reproj_args* a) { return a && reproj_launch(*a, b200()).finalizes_itself ? 1 : 0; }

int emu_reproj_finalize(const bbd_reproj_args* ap, float* loss, float* gpose) {
  const bbd_reproj_args& a = *ap;
  const ReprojLaunch L = reproj_launch(a, b200());
  const int ntiles = L.stride, used = L.used, used_grad = L.used_grad;
  for (int s = 0; s < a.num_scales; ++s) {
    float tot = 0.0f;
    for (int i = 0; i < a.batch * used; ++i) tot += a.loss_part[(size_t)s * a.batch * ntiles + (size_t)(i / used) * ntiles + (i % used)];
    loss[s] = tot / ((float)a.batch * (float)a.height * (float)a.width);
  }
  if (!gpose) return 0;
  for (int s = 0; s < a.num_scales; ++s)
    for (int pose = 0; pose < a.num_pose; ++pose)
      for (int c = 0; c < 12; ++c) {
        float acc = 0.0f;
        for (int b = 0; b < a.batch; ++b) {
          const int n_rep = a.tab.hdr[(size_t)b * 4];
          for (int k = 0; k < n_rep; ++k) {
            if (a.tab.rep[((size_t)b * BBD_MAX_REP + k) * 4 + 2] != pose) continue;
            const float* p = a.gpose_part + (((size_t)s * a.batch + b) * BBD_MAX_REP + k) * ntiles * 12;
            for (int tI = 0; tI < used_grad; ++tI) acc += p[(size_t)tI * 12 + c];
          }
        }
        gpose[((size_t)s * a.num_pose + pose) * 12 + c] = acc;
      }
  return 0;
}

size_t emu_smooth_scratch_floats(int32_t batch, int32_t levels, const int32_t* h, const int32_t* w) {
  return smooth_layout(batch, levels, h, w).floats;
}

int emu_smooth_fused(const bbd_smooth_args* in) {
  bbd_smooth_args a = *in;
  const SmoothLayout lay = smooth_layout(a.batch, a.levels, a.h, a.w);
  a.max_chunks = lay.max_parts;
  float* coef = a.defer_norm ? a.coef : a.scratch + lay.scalars;
  // stage 2: one fiber block per warp of the device kernel's blocks
  for (int lvl = 0; lvl < a.levels; ++lvl)
    for (int b = 0; b < a.batch; ++b) {
      const int nbx = smr_nbx(a.w[lvl]), nby = smr_nby(a.h[lvl]);
      for (int by = 0; by < nby; ++by)
        for (int bx = 0; bx < nbx; ++bx) {
          float tot[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          for (int warp = 0; warp < SMR_WARPS; ++warp) {
            float out[4];
            simt::run_block(32, [&](int tid) {
              float o[4];
              sm_rows_lane(a, lvl, b, bx, by, warp, tid, o);
              if (tid == 0) { out[0] = o[0]; out[1] = o[1]; out[2] = o[2]; out[3] = o[3]; }
            });
            for (int k = 0; k < 4; ++k) tot[k] += out[k];
          }
          for (int k = 0; k < 4; ++k) sm_slot(a, lvl, b, k < 3 ? 1 + k : 0)[by * nbx + bx] = tot[k];
        }
    }
  std::vector<float> tx(a.levels * a.batch), ty(a.levels * a.batch);
  for (int i = 0; i < a.levels * a.batch; ++i) {
    float sums[2];
    sm_finish_sample(a, i / a.batch, i % a.batch, coef, sums);
    tx[i] = sums[0];
    ty[i] = sums[1];
  }
  for (int lvl = 0; lvl < a.levels; ++lvl) a.loss[lvl] = sm_level_loss(a, lvl, tx.data() + lvl * a.batch, ty.data() + lvl * a.batch);
  if (!a.defer_norm && a.normalize)
    for (int lvl = 0; lvl < a.levels; ++lvl)
      if (a.gdisp[lvl])
        for (int b = 0; b < a.batch; ++b)
          for (int i = 0; i < a.h[lvl] * a.w[lvl]; ++i) sm_apply_px(a, coef, lvl, b, i);
  return 0;
}

// four pixels of a row per thread, stored as the device kernel stores them (one float4 where d2d_forward_vec allows)
int emu_disp_to_depth_forward(const bbd_d2d_args* ap) {
  const bbd_d2d_args& a = *ap;
  const int H = a.height, W = a.width;
  const bool vec = d2d_forward_vec(a);
  for (int lvl = 0; lvl < a.levels; ++lvl) {
    const float sy = (float)a.h[lvl] / (float)H, sx = (float)a.w[lvl] / (float)W;
    for (int row = 0; row < a.batch * H; ++row)
      for (int x4 = 0; x4 < W; x4 += 4) {
        float v[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        for (int k = 0; k < 4 && x4 + k < W; ++k) v[k] = d2d_forward_px(a, lvl, row / H, row % H, x4 + k, sy, sx);
        float* o = a.depth + ((size_t)lvl * a.batch * H + row) * W + x4;
        if (vec) st4g(o, v[0], v[1], v[2], v[3]);
        else
          for (int k = 0; k < 4 && x4 + k < W; ++k) o[k] = v[k];
      }
  }
  return 0;
}

size_t emu_d2d_scratch_floats(const bbd_d2d_args* a) { return d2d_scratch_offset(*a, a->levels); }

int emu_disp_to_depth_backward_pass1(const bbd_d2d_args* ap) {
  const bbd_d2d_args& a = *ap;
  if (a.scratch)
    for (int lvl = 0; lvl < a.levels; ++lvl) {
      const int f = d2d_sep_factor(a, lvl);
      if (!f) continue;
      const int w = a.w[lvl], H = a.height;
      float* tmp = a.scratch + d2d_scratch_offset(a, lvl);
      for (int i = 0; i < a.batch * H * w; ++i) {
        const int ix = i % w, r = i / w, oy = r % H, b = r / H;
        tmp[i] = f == 2 ? d2d_hpass<2>(a, lvl, b, oy, ix) : (f == 4 ? d2d_hpass<4>(a, lvl, b, oy, ix) : d2d_hpass<8>(a, lvl, b, oy, ix));
      }
    }
  return 0;
}

int emu_disp_to_depth_backward_pass2(const bbd_d2d_args* ap, int32_t level_begin, int32_t level_end) {
  const bbd_d2d_args& a = *ap;
  for (int lvl = level_begin; lvl < level_end; ++lvl) {
    const int h = a.h[lvl], w = a.w[lvl];
    const float sy = (float)h / (float)a.height, sx = (float)w / (float)a.width;
    for (int b = 0; b < a.batch; ++b)
      for (int i = 0; i < h * w; ++i) a.gdisp[lvl][(size_t)b * h * w + i] = d2d_backward_px(a, lvl, b, i / w, i % w, sy, sx);
  }
  return 0;
}

}  // extern "C"
template <int F>
static void emu_d2d_fused_level(const bbd_d2d_args& a, int lvl) {
  std::vector<float> srow(a.width);
  for (int b = 0; b < a.batch; ++b)
    for (int iy = 0; iy < a.h[lvl]; ++iy) {
      if (F == 1) {  // same resolution: four columns per thread, one float4 store (d2d_backward_fused_kernel)
        const size_t row = (size_t)b * a.h[lvl] + iy;
        for (int x4 = 0; x4 < a.width; x4 += 4) {
          float v[4];
          d2d_fused_col4<1>(a, lvl, b, iy, x4, v);
          for (int j = 0; j < 4; ++j) v[j] = d2d_epilogue(a, lvl, b, iy, x4 + j, v[j]);
          st4g(a.gdisp[lvl] + row * a.w[lvl] + x4, v[0], v[1], v[2], v[3]);
        }
        continue;
      }
      for (int x4 = 0; x4 < a.width; x4 += 4) d2d_fused_col4<F>(a, lvl, b, iy, x4, srow.data() + x4);
      for (int ix = 0; ix < a.w[lvl]; ++ix)
        a.gdisp[lvl][((size_t)b * a.h[lvl] + iy) * a.w[lvl] + ix] = d2d_fused_out<F>(a, lvl, b, iy, ix, srow.data());
    }
}
extern "C" {
int emu_disp_to_depth_backward(const bbd_d2d_args* ap) {
  const bbd_d2d_args& a = *ap;
  if (d2d_single_launch(a)) {
    for (int l = 0; l < a.levels; ++l) {
      const int f = d2d_fused_factor(a, l);
      if (f == 1) emu_d2d_fused_level<1>(a, l);
      else if (f == 2) emu_d2d_fused_level<2>(a, l);
      else if (f == 4) emu_d2d_fused_level<4>(a, l);
      else emu_d2d_fused_level<8>(a, l);
    }
    return 0;
  }
  emu_disp_to_depth_backward_pass1(ap);
  return emu_disp_to_depth_backward_pass2(ap, 0, ap->levels);
}

int emu_pose_forward(int32_t n, const float* aa, const float* tr, int32_t invert, float* T) {
  for (int i = 0; i < n; ++i) pose_forward_one(aa + (size_t)i * 3, tr + (size_t)i * 3, invert, T + (size_t)i * 16);
  return 0;
}
int emu_pose_backward(int32_t n, const float* aa, const float* tr, int32_t invert, const float* gT, float* gaa, float* gtr) {
  for (int i = 0; i < n; ++i)
    pose_backward_one(aa + (size_t)i * 3, tr + (size_t)i * 3, invert, gT + (size_t)i * 16, gaa + (size_t)i * 3, gtr + (size_t)i * 3);
  return 0;
}

int emu_pose_pack_forward(int32_t n, const float* K, const int32_t* k_row, const float* T, float* P) {
  for (int i = 0; i < n * 12; ++i)
    P[i] = pose_pack_elem(K + (size_t)k_row[i / 12] * 16, T + (size_t)(i / 12) * 16, (i % 12) / 4, i % 4);
  return 0;
}
int emu_pose_pack_backward(int32_t n, const float* K, const int32_t* k_row, const float* gP, float* gT) {
  for (int i = 0; i < n * 16; ++i)
    gT[i] = pose_pack_grad_elem(K + (size_t)k_row[i / 16] * 16, gP + (size_t)(i / 16) * 12, (i % 16) / 4, i % 4);
  return 0;
}

int emu_warp_forward(int32_t n, int32_t H, int32_t W, const float* images, const float* depth, const float* inv_K,
                     const float* P, float* warped, float* grid) {
  for (int b = 0; b < n; ++b)
    for (int i = 0; i < H * W; ++i) warp_px(H, W, images, depth, inv_K, P, b, i / W, i % W, warped, grid);
  return 0;
}

int emu_backproject_forward(int32_t n, int32_t H, int32_t W, const float* depth, const float* inv_K, float* points) {
  for (int b = 0; b < n; ++b)
    for (int i = 0; i < H * W; ++i) backproject_px(H * W, W, depth, inv_K, b, i, points);
  return 0;
}
int emu_backproject_backward(int32_t n, int32_t H, int32_t W, const float* inv_K, const float* gpoints, float* gdepth) {
  for (int b = 0; b < n; ++b)
    for (int i = 0; i < H * W; ++i) gdepth[(size_t)b * H * W + i] = backproject_grad_px(H * W, W, inv_K, gpoints, b, i);
  return 0;
}
int emu_project_forward(int32_t n, int32_t H, int32_t W, const float* points, const float* P, float eps, float* pix) {
  for (int b = 0; b < n; ++b)
    for (int i = 0; i < H * W; ++i) project_px(H, W, points, P, eps, b, i, pix);
  return 0;
}
int emu_project_chunks(int32_t, int32_t) { return 1; }
int emu_project_backward(int32_t n, int32_t H, int32_t W, const float* points, const float* P, float eps, const float* gpix,
                         float* gpoints, float* gP_part) {
  for (int b = 0; b < n; ++b) {
    float gP[12] = {0};
    for (int i = 0; i < H * W; ++i) project_grad_px(H, W, points, P, eps, gpix, b, i, gpoints, gP);
    for (int k = 0; k < 12; ++k) gP_part[(size_t)b * 12 + k] = gP[k];
  }
  return 0;
}
int emu_grid_sample_forward(int32_t n, int32_t C, int32_t H, int32_t W, int32_t Ho, int32_t Wo, const float* images,
                            const float* grid, float* out) {
  for (int b = 0; b < n; ++b)
    for (int o = 0; o < Ho * Wo; ++o) grid_sample_px(C, H, W, Ho * Wo, images, grid, b, o, out);
  return 0;
}
int emu_grid_sample_dest_keys(int32_t n, int32_t H, int32_t W, int32_t Ho, int32_t Wo, const float* grid, int32_t* keys) {
  for (int b = 0; b < n; ++b)
    for (int o = 0; o < Ho * Wo; ++o) keys[(size_t)b * Ho * Wo + o] = gs_dest_key(H, W, Ho * Wo, grid, b, o);
  return 0;
}
int emu_grid_sample_backward_image(int32_t n, int32_t C, int32_t H, int32_t W, int32_t Ho, int32_t Wo, const float* grid,
                                   const float* gout, const int32_t* keys_sorted, const int32_t* order, int32_t* seg_start,
                                   float* gimages) {
  const int n_items = n * Ho * Wo, n_keys = n * H * W;
  for (int i = 0; i <= n_items; ++i) gs_segment_mark(keys_sorted, n_items, n_keys, i, seg_start);
  for (int b = 0; b < n; ++b)
    for (int c = 0; c < C; ++c)
      for (int p = 0; p < H * W; ++p)
        gimages[((size_t)b * C + c) * H * W + p] = gs_image_grad_px(C, H, W, Ho * Wo, grid, gout, seg_start, order, b, c, p);
  return 0;
}
int emu_grid_sample_backward(int32_t n, int32_t C, int32_t H, int32_t W, int32_t Ho, int32_t Wo, const float* images,
                             const float* grid, const float* gout, float* ggrid) {
  for (int b = 0; b < n; ++b)
    for (int o = 0; o < Ho * Wo; ++o) grid_sample_grad_px(C, H, W, Ho * Wo, images, grid, gout, b, o, ggrid);
  return 0;
}

int emu_ssim_forward(int32_t n, int32_t ch, int32_t H, int32_t W, const float* x, const float* y, float* out) {
  for (size_t pl = 0; pl < (size_t)n * ch; ++pl)
    for (int i = 0; i < H * W; ++i) out[pl * H * W + i] = ssim_px(x + pl * H * W, y + pl * H * W, H, W, i / W, i % W);
  return 0;
}
int emu_ssim_backward(int32_t n, int32_t ch, int32_t H, int32_t W, const float* x, const float* y, const float* gout,
                      float* gx, float* gy) {
  for (size_t pl = 0; pl < (size_t)n * ch; ++pl)
    for (int i = 0; i < H * W; ++i)
      ssim_grad_px(x + pl * H * W, y + pl * H * W, gout + pl * H * W, H, W, i / W, i % W, gx ? gx + pl * H * W : nullptr,
                   gy ? gy + pl * H * W : nullptr);
  return 0;
}

int emu_loss_combine_forward(int32_t n, const float* reproj, const float* smooth, const float* weight, float num_scales,
                             float* per_scale, float* total) {
  loss_combine(n, reproj, smooth, weight, num_scales, per_scale, total);
  return 0;
}
int emu_loss_combine_backward(int32_t n, const float* g_total, const float* g_per_scale, const float* weight,
                              float num_scales, float* g_reproj, float* g_smooth) {
  loss_combine_grad(n, g_total, g_per_scale, weight, num_scales, g_reproj, g_smooth);
  return 0;
}

int emu_u8_to_f32(const uint8_t* src, float* dst, size_t n) {
  for (size_t i = 0; i < n; ++i) dst[i] = u8_to_unit(src[i]);
  return 0;
}

// gradients w.r.t. the colour frames (bbd_framegrad.cuh), one pixel at a time
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
