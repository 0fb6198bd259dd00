// libbbd_loss.so: sm_100a kernels and the C ABI declared in include/bbd_loss.h.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
// (see baseboostdepth_b200/build.py).  No torch types cross this file's boundary.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <string.h>

#include "bbd_ops.cuh"
#include "bbd_smooth.cuh"
#include "bbd_strip.cuh"
#include "bbd_stream.cuh"
#include "bbd_pipe.cuh"
#include "bbd_framegrad.cuh"

namespace bbd {

// Identity pre-pass and fused loss share one tile geometry: 28x16 target pixels per block of 6
// warps, lanes = columns (bbd_strip.cuh).  With two warped candidates a block needs 64 KB of shared
// memory -> 3 blocks (18 warps) per SM at 96 registers per thread.  Fewer, fatter warps beat 8 warps
// at 80 registers: the kernel gains from instruction-level parallelism inside a warp (four rows of
// gathers in flight in the warp phase, two rows walked together in the backward), not from more
// resident warps (profiles/README.md lists the measured variants).
#ifndef BBD_TILE_H
#define BBD_TILE_H 16
#endif
#ifndef BBD_MIN_BLOCKS
#define BBD_MIN_BLOCKS 3
#endif
#ifndef BBD_WARPS
#define BBD_WARPS 6
#endif
#ifndef BBD_SCATTER_REDUCE
#define BBD_SCATTER_REDUCE 1
#endif
using SCfg = StripCfg<BBD_TILE_H, BBD_WARPS>;

static thread_local char g_err[256] = "";

static int fail(int code, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s", what);
  return code;
}
static int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// identity pre-pass
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SCfg::NT) ident_kernel(const bbd_ident_args a) {
  extern __shared__ float smem[];
  IdentStripSmem<SCfg> sm;
  sm.carve(smem);
  const int tid = threadIdx.x;
  const StripCtx t = make_strip<SCfg>(blockIdx.x, blockIdx.y, blockIdx.z, tid, a.batch, a.height, a.width);
  const int H = a.height, W = a.width;
  const int32_t* hdr = a.tab.hdr + (size_t)t.b * 4;
  const int n_id = hdr[1];
  const float* noise = a.noise[hdr[2]] + (size_t)hdr[3] * H * W;
  is_load<SCfg>(a.target + (size_t)t.b * 3 * H * W, sm.tgt, t, H, W);
  __syncthreads();
  is_target_stats<SCfg>(a, sm, t);
  for (int j = 0; j < n_id; ++j) {
    const int32_t* e = a.tab.ident + ((size_t)t.b * BBD_MAX_IDENT + j) * 2;
    is_load<SCfg>(a.frames[e[0]] + (size_t)e[1] * 3 * H * W, sm.src, t, H, W);
    __syncthreads();
    is_candidate<SCfg>(a, sm, t, j, noise);
    __syncthreads();
  }
  is_store<SCfg>(a, sm, t);
}

// ------------------------------------------------------------------------------------------
// fused reprojection loss
// ------------------------------------------------------------------------------------------
// Block sum of K per-thread values in a fixed order: xor-butterfly inside each warp, then the NW
// warp partials are added by one thread per component.  No atomics.  red: [NW][12] floats.
template <int K>
__device__ __forceinline__ void block_reduce(float* red, int tid, const float* v, float* out) {
#if BBD_SCATTER_REDUCE
  if (K == 12) {
    // Reduce-scatter over the warp: at every step a lane hands one half of its values to its partner
    // and adds the partner's other half, so 16 shuffles (instead of 60) leave component (lane >> 1)
    // summed over the warp in r[0].  Fixed order: deterministic.
    const int lane = tid & 31;
    float r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) r[i] = i < K ? v[i] : 0.0f;
#pragma unroll
    for (int n = 8, off = 16; n >= 1; n >>= 1, off >>= 1) {
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < n; ++i) {
        const float send = upper ? r[i] : r[i + n];
        const float keep = upper ? r[i + n] : r[i];
        r[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
    r[0] += __shfl_xor_sync(0xffffffffu, r[0], 1);
    const int comp = lane >> 1;
    if ((lane & 1) == 0 && comp < K) red[(tid >> 5) * 12 + comp] = r[0];
  } else
#endif
  {
    float r[K];
#pragma unroll
    for (int i = 0; i < K; ++i) r[i] = v[i];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
      for (int i = 0; i < K; ++i) r[i] += __shfl_xor_sync(0xffffffffu, r[i], off);
    }
    if ((tid & 31) == 0) {
#pragma unroll
      for (int i = 0; i < K; ++i) red[(tid >> 5) * 12 + i] = r[i];
    }
  }
  __syncthreads();
  if (tid < K) {
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < SCfg::NW; ++w) s += red[w * 12 + tid];
    out[tid] = s;
  }
  __syncthreads();
}

// grid (tiles_x, tiles_y, S*B): one block per tile of one (scale, sample).  (Walking over the four
// scales inside one block to share the target tile was measured slower: 4x fewer blocks, more
// live state -> spills at 80 registers.)
// KEEP: one warped tile per candidate stays in shared memory (fastest for <= 2 candidates);
// otherwise a single tile buffer is reused and the backward recomputes the warped value.
template <bool GRAD, bool KEEP>
__global__ void __launch_bounds__(SCfg::NT, BBD_MIN_BLOCKS) reproj_kernel(const bbd_reproj_args a) {
  extern __shared__ float smem[];
  StripSmem<SCfg> sm;
  sm.carve(smem, KEEP ? a.max_rep : 1);
  const int tid = threadIdx.x;
  const StripCtx t = make_strip<SCfg>(blockIdx.x, blockIdx.y, blockIdx.z, tid, a.batch, a.height, a.width);
  const int n_rep = a.tab.hdr[(size_t)t.b * 4];

  rs_load_target<SCfg>(a, sm, t, tid);  // asynchronous copies, in flight during the first warp phase
  rs_begin_scale<SCfg>(sm, tid);
  {
    for (int k = 0; k < n_rep; ++k) {
      if (!KEEP && k) __syncthreads();  // the single warped-tile buffer is reused by every candidate
      rs_warp<SCfg, KEEP>(a, sm, t, k);
      if (k == 0) rs_load_wait();
      __syncthreads();
      if (k == 0) rs_target_stats<SCfg>(a, sm, t);  // each thread reads back only slots it wrote itself
      rs_stats<SCfg, KEEP>(a, sm, t, k);
    }
    if (n_rep == 0) {  // no warped candidate at all: the identity minimum wins everywhere
      rs_load_wait();
      __syncthreads();
    }
    const float part = rs_select<SCfg>(a, sm, t, n_rep);
    block_reduce<1>(sm.red, tid, &part, a.loss_part + ((size_t)t.s * a.batch + t.b) * t.ntiles + t.tile);

    if (GRAD) {
      for (int k = 0; k < BBD_MAX_REP; ++k) {
        float* out = a.gpose_part + ((((size_t)t.s * a.batch + t.b) * BBD_MAX_REP + k) * t.ntiles + t.tile) * 12;
        if (k >= n_rep || !sm.anywin[k]) {  // block-uniform
          if (tid < 12) out[tid] = 0.0f;
          continue;
        }
        float gP[12];
        {
          const float* src;
          Cam cam;
          rs_candidate(a, t.b, k, src, cam);
#pragma unroll
          for (int i = 0; i < 12; ++i) gP[i] = 0.0f;
          for (int q = t.warp; q < SCfg::TH; q += BBD_BWD_ROWS * SCfg::NW) {  // warp-uniform
#pragma unroll
            for (int r = 0; r < BBD_BWD_ROWS; ++r)
              if (q + r * SCfg::NW < SCfg::TH) rs_bwd_vertical<SCfg>(a, sm, t, k, q + r * SCfg::NW, r);
            __syncwarp();
#pragma unroll
            for (int r = 0; r < BBD_BWD_ROWS; ++r)
              if (q + r * SCfg::NW < SCfg::TH) rs_bwd_horizontal<SCfg, KEEP>(a, sm, t, k, q + r * SCfg::NW, src, cam, gP, r);
            __syncwarp();
          }
        }
        block_reduce<12>(sm.red, tid, gP, out);
      }
      rs_store_gdepth<SCfg>(a, sm, t);
    }
  }
}


// ------------------------------------------------------------------------------------------
// fused reprojection loss, streaming form (bbd_stream.cuh): one warp = one strip segment
// ------------------------------------------------------------------------------------------
#ifndef BBD_STREAM_WARPS
#define BBD_STREAM_WARPS 1  // one warp per block: every branch on the unit index is provably warp-uniform,
                            // so the shuffles need no WARPSYNC / ENDCOLLECTIVE brackets
#endif
#ifndef BBD_STREAM_MINB
#define BBD_STREAM_MINB 8
#endif
template <int K, bool GRAD, bool MULTI, bool WING = false>
__global__ void __launch_bounds__(BBD_STREAM_WARPS * 32, BBD_STREAM_MINB) reproj_stream_kernel(const bbd_reproj_args a, int n_units, int part_stride, int seg_rows) {
  extern __shared__ __align__(128) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * BBD_STREAM_WARPS + warp;
  if (unit >= n_units) return;  // warp-uniform
  StreamTmaMaps none = {nullptr, nullptr, nullptr};
  stream_unit<K, GRAD, false, MULTI, WING>(a, unit, lane, smem + (size_t)warp * StreamSmem<K, false, MULTI, GRAD, MULTI && !WING>::FLOATS, part_stride, none, seg_rows);
}

// The same kernel with the strip's regular planes (target, depth, identity minimum) staged by the TMA unit.
template <int K, bool GRAD, bool MULTI, bool WING = false>
__global__ void __launch_bounds__(BBD_STREAM_WARPS * 32, BBD_STREAM_MINB)
    reproj_stream_tma_kernel(const bbd_reproj_args a, int n_units, int part_stride, const __grid_constant__ CUtensorMap tm_tgt,
                             const __grid_constant__ CUtensorMap tm_dep, const __grid_constant__ CUtensorMap tm_idm, int seg_rows) {
  extern __shared__ __align__(128) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x * BBD_STREAM_WARPS + warp;
  if (unit >= n_units) return;  // warp-uniform
  StreamTmaMaps maps = {&tm_tgt, &tm_dep, &tm_idm};
  stream_unit<K, GRAD, true, MULTI, WING>(a, unit, lane, smem + (size_t)warp * StreamSmem<K, true, MULTI, GRAD, MULTI && !WING>::FLOATS, part_stride, maps, seg_rows);
}

// The pipelined form (bbd_pipe.cuh): one block = one unit, its warps are the gather / statistics / backward
// stages of the row program.  128 registers per thread -> five blocks (15 warps) per SM.
#ifndef BBD_PIPE_MINB
#define BBD_PIPE_MINB 5
#endif
template <int K, bool GRAD>
__global__ void __launch_bounds__(GRAD ? 96 : 64, BBD_PIPE_MINB)
    reproj_pipe_kernel(const bbd_reproj_args a, int n_units, int part_stride, const __grid_constant__ CUtensorMap tm_tgt,
                       const __grid_constant__ CUtensorMap tm_dep, const __grid_constant__ CUtensorMap tm_idm, int seg_rows) {
  extern __shared__ __align__(128) float smem[];
  const int unit = blockIdx.x;
  if (unit >= n_units) return;  // block-uniform
  StreamTmaMaps maps = {&tm_tgt, &tm_dep, &tm_idm};
  pipe_unit<K, GRAD>(a, unit, threadIdx.x, smem, part_stride, maps, seg_rows);
}

__global__ void stream_coords_kernel(int n, int H, int W, const float* depth, const float* inv_K, const float* P, float* grid,
                                     float* pix) {
  const size_t total = (size_t)n * H * W;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    stream_coords_px(H, W, depth, inv_K, P, (int)(i / ((size_t)H * W)), (int)((i / W) % H), (int)(i % W), grid, pix);
}

// identity pre-pass, streaming form: one warp per block = one strip segment of one sample
struct RgbaPtrs {
  float* p[BBD_MAX_FRAMES];
};
__global__ void __launch_bounds__(32) ident_stream_kernel(const bbd_ident_args a, const RgbaPtrs rgba, int n_units, int seg_rows) {
  const int unit = blockIdx.x;
  if (unit >= n_units) return;
  ident_unit(a, rgba.p, unit, threadIdx.x, seg_rows);
}

// (n,3,H,W) -> (n,H,W,4): a thread converts four consecutive pixels (3 x 16 B in, 4 x 16 B out)
__global__ void __launch_bounds__(256) pack_rgba_kernel(int n, int HW, const float* __restrict__ planar, float4* __restrict__ rgba) {
  const int q = HW / 4;  // HW % 4 == 0 is checked by the launcher for this path
  const size_t total = (size_t)n * q;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t img = i / q, j = i - img * q;
    const float4* p = reinterpret_cast<const float4*>(planar + img * 3 * HW) + j;
    const float4 r = p[0], g = p[q], b = p[2 * (size_t)q];
    float4* o = rgba + img * HW + j * 4;
    o[0] = make_float4(r.x, g.x, b.x, 0.0f);
    o[1] = make_float4(r.y, g.y, b.y, 0.0f);
    o[2] = make_float4(r.z, g.z, b.z, 0.0f);
    o[3] = make_float4(r.w, g.w, b.w, 0.0f);
  }
}
__global__ void __launch_bounds__(256) pack_rgba_scalar_kernel(int n, int HW, const float* __restrict__ planar, float4* __restrict__ rgba) {
  const size_t total = (size_t)n * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t img = i / HW, j = i - img * HW;
    const float* p = planar + img * 3 * HW + j;
    rgba[i] = make_float4(p[0], p[HW], p[2 * (size_t)HW], 0.0f);
  }
}

// Sum the per-tile partials in a fixed order.  grid.x = S * (1 + num_pose); block 0..S-1 -> loss.
// 768 threads = 64 tile-lanes x 12 components: every thread adds its share of the partials, a
// fixed-order tail adds the lanes (deterministic, no atomics).
constexpr int FIN_NT = 768, FIN_LANES = FIN_NT / 12;
__global__ void __launch_bounds__(FIN_NT) reproj_finalize_kernel(const bbd_reproj_args a, float* loss, float* gpose, int ntiles, int used, int used_grad) {
  __shared__ float red[FIN_NT];
  __shared__ float red2[32];
  const int tid = threadIdx.x;
  const int S = a.num_scales;
  if ((int)blockIdx.x < S) {
    const int s = blockIdx.x;
    const float* p = a.loss_part + (size_t)s * a.batch * ntiles;
    float acc = 0.0f;
    if (used == ntiles) {
      for (int i = tid; i < a.batch * ntiles; i += FIN_NT) acc += p[i];
    } else {
      for (int i = tid; i < a.batch * used; i += FIN_NT) acc += p[(i / used) * ntiles + (i % used)];
    }
    red[tid] = acc;
    __syncthreads();
    if (tid < 32) {
      float part = 0.0f;
      for (int i = 0; i < FIN_NT / 32; ++i) part += red[tid * (FIN_NT / 32) + i];
      red2[tid] = part;
    }
    __syncthreads();
    if (tid == 0) {
      float tot = 0.0f;
      for (int i = 0; i < 32; ++i) tot += red2[i];
      loss[s] = tot / ((float)a.batch * (float)a.height * (float)a.width);
    }
    return;
  }
  if (!gpose) return;
  // one block per (scale, pose row): find the (sample, candidate) pairs that use this pose
  const int idx = blockIdx.x - S, s = idx / a.num_pose, pose = idx % a.num_pose;
  const int comp = tid % 12, lane = tid / 12;
  float acc = 0.0f;
  for (int b = 0; b < a.batch; ++b) {
    const int n_rep = a.tab.hdr[(size_t)b * 4];
    for (int k = 0; k < n_rep; ++k) {
      if (a.tab.rep[((size_t)b * BBD_MAX_REP + k) * 4 + 2] != pose) continue;
      const float* p = a.gpose_part + (((size_t)s * a.batch + b) * BBD_MAX_REP + k) * ntiles * 12;
      for (int tI = lane; tI < used_grad; tI += FIN_LANES) acc += p[(size_t)tI * 12 + comp];
    }
  }
  red[tid] = acc;
  __syncthreads();
  if (tid < 12) {
    float tot = 0.0f;
    for (int l = 0; l < FIN_LANES; ++l) tot += red[l * 12 + tid];
    gpose[((size_t)s * a.num_pose + pose) * 12 + tid] = tot;
  }
}

// ------------------------------------------------------------------------------------------
// smoothness
// ------------------------------------------------------------------------------------------
// grid (column blocks, row chunks, levels * B); 4 warps x 30 owned columns per block.  The last block to
// take a ticket reduces the partials (fixed order) to the level losses and the per-sample scalars.
__global__ void __launch_bounds__(SMR_WARPS * 32) smooth_rows_kernel(const SmoothArgs a, float* coef, unsigned* ticket, unsigned total) {
  __shared__ float red[SMR_WARPS][4];
  __shared__ int last_s;
  __shared__ float tx_s[BBD_MAX_SCALES * 256], ty_s[BBD_MAX_SCALES * 256];
  const int lvl = blockIdx.z / a.batch, b = blockIdx.z - lvl * a.batch, bx = blockIdx.x, by = blockIdx.y;
  const int nbx = smr_nbx(a.w[lvl]);
  if (bx >= nbx || by >= smr_nby(a.h[lvl])) return;  // block-uniform
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float out[4];
  sm_rows_lane(a, lvl, b, bx, by, warp, lane, out);
  if (lane == 0) { red[warp][0] = out[0]; red[warp][1] = out[1]; red[warp][2] = out[2]; red[warp][3] = out[3]; }
  __syncthreads();
  if (tid == 0) {
    const int slot = by * nbx + bx;
    for (int k = 0; k < 4; ++k) {
      float v = 0.0f;
      for (int w = 0; w < SMR_WARPS; ++w) v += red[w][k];
      sm_slot(a, lvl, b, k < 3 ? 1 + k : 0)[slot] = v;  // slots 1..3: loss and coupling sums, slot 0: sum of the disparity
    }
    __threadfence();
    last_s = (atomicAdd(ticket, 1u) == total - 1u) ? 1 : 0;
  }
  __syncthreads();
  if (!last_s) return;
  __threadfence();
  const int pairs = a.levels * a.batch;
  for (int i = tid; i < pairs; i += blockDim.x) {
    float sums[2];
    sm_finish_sample(a, i / a.batch, i % a.batch, coef, sums);
    tx_s[i] = sums[0];
    ty_s[i] = sums[1];
  }
  __syncthreads();
  if (tid < a.levels) a.loss[tid] = sm_level_loss(a, tid, tx_s + tid * a.batch, ty_s + tid * a.batch);
  if (tid == 0) *ticket = 0u;  // ready for the next launch
}

__global__ void __launch_bounds__(256) smooth_apply_kernel(const SmoothArgs a, const float* coef) {
  const int lvl = blockIdx.z, b = blockIdx.y;
  const int n = a.h[lvl] * a.w[lvl];
  if (!a.gdisp[lvl]) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) sm_apply_px(a, coef, lvl, b, i);
}

// ------------------------------------------------------------------------------------------
// element-wise operators
// ------------------------------------------------------------------------------------------
// grid (blocks, 1, levels): the per-level interpolation scales are block constants.  A thread
// produces four consecutive pixels of a row (one 16-byte store when the row pitch allows), sharing
// the row taps.
// grid (column blocks, row groups, levels): a thread owns four consecutive columns, whose source
// taps it computes once, and walks rows (b, py); no per-thread division, float4 stores.
__global__ void __launch_bounds__(128) d2d_forward_kernel(const bbd_d2d_args a) {
  const int lvl = blockIdx.z;
  const int H = a.height, W = a.width, HW = H * W;
  const int h = a.h[lvl], w = a.w[lvl];
  const int gw = (W + 3) / 4;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= gw) return;
  const float sy = div_((float)h, (float)H), sx = div_((float)w, (float)W);
  float* out = a.depth + (size_t)lvl * a.batch * HW;
  const bool vec = (W % 4) == 0;
  const bool same = (h == H && w == W);  // taps are (o, o) with weights (1, 0): the value itself
  Lerp tx[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) tx[k] = up_taps(min(g * 4 + k, W - 1), w, sx);
  for (int row = blockIdx.y; row < a.batch * H; row += gridDim.y) {
    const int b = row / H, py = row - b * H;
    const float* d = a.disp[lvl] + (size_t)b * h * w;
    const Lerp ty = up_taps(py, h, sy);
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int px = g * 4 + k;
      if (px < W) {
        const float up = same ? d[py * W + px] : d2d_up(d, w, ty, tx[k]);
        v[k] = a.sql ? up : rcp_rn(add(a.min_disp, mul(a.disp_span, up)));
      } else {
        v[k] = 0.0f;
      }
    }
    float* o = out + (size_t)row * W + g * 4;
    if (vec) {
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (g * 4 + k < W) o[k] = v[k];
    }
  }
}

// grid (column blocks, row blocks, levels): a block walks full-resolution rows (b, oy), its threads
// are low-resolution columns -- no per-thread division, row-contiguous loads and stores.  (A
// vertical-first streaming pass with one thread per full-resolution column, every row read once
// and coalesced, was measured slower: 40 us against 29 us.)
__global__ void __launch_bounds__(128) d2d_hpass_kernel(const bbd_d2d_args a) {
  const int lvl = blockIdx.z;
  const int f = d2d_sep_factor(a, lvl);
  if (!f) return;
  const int w = a.w[lvl], H = a.height;
  const int ix = blockIdx.x * blockDim.x + threadIdx.x;
  if (ix >= w) return;
  float* tmp = a.scratch + d2d_scratch_offset(a, lvl);
  for (int row = blockIdx.y; row < a.batch * H; row += gridDim.y) {
    const int b = row / H, oy = row - b * H;
    tmp[(size_t)row * w + ix] =
        f == 2 ? d2d_hpass<2>(a, lvl, b, oy, ix) : (f == 4 ? d2d_hpass<4>(a, lvl, b, oy, ix) : d2d_hpass<8>(a, lvl, b, oy, ix));
  }
}

// grid (column blocks, rows, levels): rows are (b, iy) of the level's own resolution
__global__ void __launch_bounds__(128) d2d_backward_kernel(const bbd_d2d_args a, int level_begin) {
  const int lvl = blockIdx.z + level_begin;
  const int h = a.h[lvl], w = a.w[lvl];
  const int ix = blockIdx.x * blockDim.x + threadIdx.x;
  if (ix >= w) return;
  const float sy = div_((float)h, (float)a.height), sx = div_((float)w, (float)a.width);
  for (int row = blockIdx.y; row < a.batch * h; row += gridDim.y) {
    const int b = row / h, iy = row - b * h;
    a.gdisp[lvl][(size_t)row * w + ix] = d2d_backward_px(a, lvl, b, iy, ix, sy, sx);
  }
}

// Single-launch backward: a persistent grid (all blocks resident) walks the list of low-resolution rows of every
// level, coarsest level first (a row of the 1/8 level reads sixteen full-resolution rows, one of the full-resolution
// level a single one), dealt round-robin so that every block gets the same mix.  Dynamic shared memory = two
// full-resolution rows of vertical tent sums (double buffer: one barrier per row).
struct D2DRowList {
  int32_t begin[BBD_MAX_SCALES + 1];  // item range of list position j
  int32_t level[BBD_MAX_SCALES];      // level at list position j
};
template <int F>
__device__ __forceinline__ void d2d_fused_row(const bbd_d2d_args& a, int lvl, int row, float* srow) {
  const int W = a.width, w = a.w[lvl], h = a.h[lvl];
  const int b = row / h, iy = row - b * h;
  if (F == 1) {  // same resolution: element-wise, 16 bytes per thread and step
    for (int x4 = threadIdx.x * 4; x4 < W; x4 += blockDim.x * 4) {
      float v[4];
      d2d_fused_col4<1>(a, lvl, b, iy, x4, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = d2d_epilogue(a, lvl, b, iy, x4 + j, v[j]);
      *reinterpret_cast<float4*>(a.gdisp[lvl] + (size_t)row * w + x4) = make_float4(v[0], v[1], v[2], v[3]);
    }
    return;
  }
  for (int x4 = threadIdx.x * 4; x4 < W; x4 += blockDim.x * 4) {
    float v[4];
    d2d_fused_col4<F>(a, lvl, b, iy, x4, v);
    *reinterpret_cast<float4*>(srow + x4) = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncthreads();
  for (int base = 0; base < w; base += blockDim.x) {  // block-uniform trip count
    const int ix = base + threadIdx.x;
    if (ix < w) a.gdisp[lvl][(size_t)row * w + ix] = d2d_fused_out<F>(a, lvl, b, iy, ix, srow);
  }
}
__global__ void __launch_bounds__(256, 3) d2d_backward_fused_kernel(const bbd_d2d_args a, const D2DRowList list) {
  extern __shared__ __align__(16) float sbuf[];
  const int total = list.begin[a.levels];
  int n = 0;
  for (int i = blockIdx.x; i < total; i += gridDim.x) {
    int j = 0;
    while (i >= list.begin[j + 1]) ++j;
    const int lvl = list.level[j], row = i - list.begin[j];
    const int f = d2d_fused_factor(a, lvl);
    float* srow = sbuf + (n & 1) * a.width;
    if (f == 1) { d2d_fused_row<1>(a, lvl, row, srow); continue; }  // no shared row used: the buffers do not advance
    if (f == 2) d2d_fused_row<2>(a, lvl, row, srow);
    else if (f == 4) d2d_fused_row<4>(a, lvl, row, srow);
    else d2d_fused_row<8>(a, lvl, row, srow);
    ++n;
  }
}

__global__ void pose_kernel(int n, const float* aa, const float* tr, int invert, float* T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) pose_forward_one(aa + (size_t)i * 3, tr + (size_t)i * 3, invert, T + (size_t)i * 16);
}
__global__ void pose_grad_kernel(int n, const float* aa, const float* tr, int invert, const float* gT, float* gaa, float* gtr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) pose_backward_one(aa + (size_t)i * 3, tr + (size_t)i * 3, invert, gT + (size_t)i * 16, gaa + (size_t)i * 3, gtr + (size_t)i * 3);
}

__global__ void pose_pack_kernel(int n, const float* K, const int32_t* k_row, const float* T, float* P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 12) return;
  const int p = i / 12, e = i % 12;
  P[i] = pose_pack_elem(K + (size_t)k_row[p] * 16, T + (size_t)p * 16, e / 4, e % 4);
}
__global__ void pose_pack_grad_kernel(int n, const float* K, const int32_t* k_row, const float* gP, float* gT) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 16) return;
  const int p = i / 16, e = i % 16;
  gT[i] = pose_pack_grad_elem(K + (size_t)k_row[p] * 16, gP + (size_t)p * 12, e / 4, e % 4);
}

__global__ void warp_kernel(int n, int H, int W, const float* images, const float* depth, const float* inv_K,
                            const float* P, float* warped, float* grid) {
  const size_t total = (size_t)n * H * W;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int px = (int)(i % W), py = (int)((i / W) % H), b = (int)(i / ((size_t)H * W));
    warp_px(H, W, images, depth, inv_K, P, b, py, px, warped, grid);
  }
}

__global__ void grid_sample_kernel(int n, int C, int H, int W, int HoWo, const float* images, const float* grid, float* out) {
  const size_t total = (size_t)n * HoWo;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    grid_sample_px(C, H, W, HoWo, images, grid, (int)(i / HoWo), (int)(i % HoWo), out);
}
__global__ void grid_sample_grad_kernel(int n, int C, int H, int W, int HoWo, const float* images, const float* grid,
                                        const float* gout, float* ggrid) {
  const size_t total = (size_t)n * HoWo;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    grid_sample_grad_px(C, H, W, HoWo, images, grid, gout, (int)(i / HoWo), (int)(i % HoWo), ggrid);
}

__global__ void gs_dest_keys_kernel(int n, int H, int W, int HoWo, const float* grid, int32_t* keys) {
  const size_t total = (size_t)n * HoWo;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    keys[i] = gs_dest_key(H, W, HoWo, grid, (int)(i / HoWo), (int)(i % HoWo));
}
__global__ void gs_segment_kernel(const int32_t* keys_sorted, int n_items, int n_keys, int32_t* seg_start) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i <= (size_t)n_items; i += (size_t)gridDim.x * blockDim.x)
    gs_segment_mark(keys_sorted, n_items, n_keys, (int)i, seg_start);
}
__global__ void gs_image_grad_kernel(int n, int C, int H, int W, int HoWo, const float* grid, const float* gout,
                                     const int32_t* seg_start, const int32_t* order, float* gimg) {
  const int HW = H * W;
  const size_t total = (size_t)n * C * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % HW), c = (int)((i / HW) % C), b = (int)(i / ((size_t)HW * C));
    gimg[i] = gs_image_grad_px(C, H, W, HoWo, grid, gout, seg_start, order, b, c, p);
  }
}

__global__ void backproject_kernel(int n, int H, int W, const float* depth, const float* inv_K, float* points) {
  const int HW = H * W;
  const size_t total = (size_t)n * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    backproject_px(HW, W, depth, inv_K, (int)(i / HW), (int)(i % HW), points);
}

__global__ void backproject_grad_kernel(int n, int H, int W, const float* inv_K, const float* gpoints, float* gdepth) {
  const int HW = H * W;
  const size_t total = (size_t)n * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    gdepth[i] = backproject_grad_px(HW, W, inv_K, gpoints, (int)(i / HW), (int)(i % HW));
}

__global__ void project_kernel(int n, int H, int W, const float* points, const float* P, float eps, float* pix) {
  const int HW = H * W;
  const size_t total = (size_t)n * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    project_px(H, W, points, P, eps, (int)(i / HW), (int)(i % HW), pix);
}

constexpr int PJ_CHUNK = 4096;
// grid (chunks, n); block 256.  gP_part (n, chunks, 12)
__global__ void __launch_bounds__(256) project_grad_kernel(int n, int H, int W, const float* points, const float* P, float eps,
                                                           const float* gpix, float* gpoints, float* gP_part) {
  __shared__ float red[12][256];
  const int HW = H * W, b = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  float gP[12];
  for (int k = 0; k < 12; ++k) gP[k] = 0.0f;
  for (int i = chunk * PJ_CHUNK + tid; i < (chunk + 1) * PJ_CHUNK && i < HW; i += 256)
    project_grad_px(H, W, points, P, eps, gpix, b, i, gpoints, gP);
  for (int k = 0; k < 12; ++k) red[k][tid] = gP[k];
  __syncthreads();
  if (tid < 12) {
    float s = 0.0f;
    for (int i = 0; i < 256; ++i) s += red[tid][i];
    gP_part[((size_t)b * gridDim.x + chunk) * 12 + tid] = s;
  }
}

__global__ void ssim_kernel(int planes, int H, int W, const float* x, const float* y, float* out) {
  const int HW = H * W;
  const size_t total = (size_t)planes * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t pl = i / HW;
    const int o = (int)(i % HW);
    out[i] = ssim_px(x + pl * HW, y + pl * HW, H, W, o / W, o % W);
  }
}

__global__ void ssim_grad_kernel(int planes, int H, int W, const float* x, const float* y, const float* gout, float* gx, float* gy) {
  const int HW = H * W;
  const size_t total = (size_t)planes * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t pl = i / HW;
    const int o = (int)(i % HW);
    ssim_grad_px(x + pl * HW, y + pl * HW, gout + pl * HW, H, W, o / W, o % W, gx ? gx + pl * HW : nullptr,
                 gy ? gy + pl * HW : nullptr);
  }
}

__global__ void loss_combine_kernel(int n, const float* reproj, const float* smooth, const float* weight, float num_scales,
                                    float* per_scale, float* total) {
  if (blockIdx.x == 0 && threadIdx.x == 0) loss_combine(n, reproj, smooth, weight, num_scales, per_scale, total);
}
__global__ void loss_combine_grad_kernel(int n, const float* g_total, const float* g_per_scale, const float* weight,
                                         float num_scales, float* g_reproj, float* g_smooth) {
  if (blockIdx.x == 0 && threadIdx.x == 0) loss_combine_grad(n, g_total, g_per_scale, weight, num_scales, g_reproj, g_smooth);
}

// 16 bytes in, 64 bytes out per thread and iteration; n16 = number of 16-byte groups
__global__ void __launch_bounds__(256) u8_to_f32_kernel(const uint4* __restrict__ src, float4* __restrict__ dst, size_t n16) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 v = src[i];
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float4 o;
      o.x = u8_to_unit((uint8_t)(w[k] & 0xff));
      o.y = u8_to_unit((uint8_t)((w[k] >> 8) & 0xff));
      o.z = u8_to_unit((uint8_t)((w[k] >> 16) & 0xff));
      o.w = u8_to_unit((uint8_t)(w[k] >> 24));
      dst[i * 4 + k] = o;
    }
  }
}
__global__ void u8_to_f32_tail_kernel(const uint8_t* src, float* dst, size_t begin, size_t n) {
  const size_t i = begin + blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) dst[i] = u8_to_unit(src[i]);
}

// Row-walking kernels: blocks along y per (column block, level).  Thousands of tiny blocks are bound
// by the block launch rate, not by their work -- a couple of row blocks per SM walk the rows instead.
#ifndef BBD_ROW_BLOCKS
#define BBD_ROW_BLOCKS 2
#endif
constexpr size_t kRowBlocks = 148 * BBD_ROW_BLOCKS;
#ifndef BBD_D2D_ROW_BLOCKS
#define BBD_D2D_ROW_BLOCKS 3
#endif

static int grid_for(size_t total, int block) {
  size_t g = (total + block - 1) / block;
  const size_t cap = 148 * 16;  // a few resident blocks per SM, grid-stride beyond that
  return (int)(g < cap ? (g ? g : 1) : cap);
}

// ------------------------------------------------------------------------------------------
// gradients w.r.t. the colour frames (bbd_framegrad.cuh): one thread per pixel, grid-stride
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) frame_grad_coef_kernel(const bbd_reproj_args a, const bbd_frame_grad_args f) {
  const int HW = a.height * a.width;
  const size_t total = (size_t)a.num_scales * a.batch * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int q = (int)(i % HW), sb = (int)(i / HW);
    fg_coef_px(a, f, sb / a.batch, sb % a.batch, q / a.width, q % a.width);
  }
}
__global__ void __launch_bounds__(256) frame_grad_pred_kernel(const bbd_reproj_args a, const bbd_frame_grad_args f) {
  const int HW = a.height * a.width;
  const size_t total = (size_t)a.batch * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % HW);
    fg_pred_px(a, f, (int)(i / HW), p / a.width, p % a.width);
  }
}
__global__ void __launch_bounds__(256) frame_grad_stack_kernel(const bbd_reproj_args a, const bbd_frame_grad_args f, int rows) {
  const int HW = a.height * a.width;
  const size_t total = (size_t)rows * 3 * HW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % HW), c = (int)((i / HW) % 3), grow = (int)(i / ((size_t)3 * HW));
    int slot, row;
    fg_locate_row(f, grow, slot, row);
    if (f.gframes[slot]) f.gframes[slot][((size_t)row * 3 + c) * HW + p] = fg_stack_px(a, f, slot, row, c, p);
  }
}
__global__ void __launch_bounds__(256) smooth_image_grad_kernel(const bbd_smooth_img_args a) {
  const int lvl = blockIdx.z, b = blockIdx.y;
  if (!a.gimg[lvl]) return;
  const int h = a.h[lvl], w = a.w[lvl], n = h * w;
  float* out = a.gimg[lvl] + (size_t)b * 3 * n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float g[3];
    smi_px(a, lvl, b, i / w, i % w, g);
    out[i] = g[0];
    out[n + i] = g[1];
    out[2 * n + i] = g[2];
  }
}

}  // namespace bbd

using namespace bbd;

static int tile_parts(int height, int width) {
  return ((width + SCfg::TW - 1) / SCfg::TW) * ((height + SCfg::TH - 1) / SCfg::TH);
}
// slots per (scale, sample) in loss_part / gpose_part: enough for either kernel
extern "C" int bbd_reproj_tiles(int32_t height, int32_t width) {
  return std::max(tile_parts(height, width), std::max(StreamGeo::strips(width) * stream_max_segs(height), StreamGeoM::units(height, width)));
}

// Which kernel serves these arguments (the finalize step must agree with the fused launch).
static bool use_stream(const bbd_reproj_args* a) {
  if (a->force_tile || a->min_rep < 1 || a->max_rep > BBD_MAX_REP) return false;
  if (BBD_STREAM_ASYNC && a->max_rep > 2) return false;
  bool any = false;
  for (int f = 0; f < BBD_MAX_FRAMES; ++f) {
    if (a->frames[f] && !a->frames_rgba[f]) return false;
    any = any || a->frames_rgba[f];
  }
  return any;
}
// resident warps of the one-warp streaming form on this device (8 per SM: 224-243 registers per thread)
static int stream_slots() {
  static int slots = 0;
  if (!slots) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    slots = sms * BBD_STREAM_MINB;
  }
  return slots;
}
static int seg_rows_for(const bbd_reproj_args* a) {
  if (a->max_rep > 2) return stream_seg_rows_uneven(a->height, a->width, a->num_scales * a->batch, stream_slots());
  return stream_seg_rows(a->height, a->width, a->num_scales * a->batch, stream_slots());
}
// The many-candidate form with gradients runs as two launches when the caller provides the winner plane: a forward-only
// selection launch (twelve warps per SM) and a gradient launch that reads the winners (tall segments).
static bool split_multi(const bbd_reproj_args* a) {
  return use_stream(a) && a->max_rep > 2 && a->need_grad && a->winner != nullptr;
}
// slots of loss_part / gpose_part a launch fills per (scale, sample): the two can differ in the split form
static int parts_used(const bbd_reproj_args* a, bool grad_parts) {
  if (!use_stream(a)) return tile_parts(a->height, a->width);
  if (a->max_rep > 2 && !(grad_parts && split_multi(a))) return StreamGeoM::units(a->height, a->width);
  const int rh = seg_rows_for(a);
  return StreamGeo::strips(a->width) * ((a->height + rh - 1) / rh);
}

#ifndef BBD_STREAM_TMA
#define BBD_STREAM_TMA (!BBD_STREAM_ASYNC)
#endif
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    cudaGetLastError();
  }
  return fn;
}
// (W, H, planes) fp32 tensor, boxes of 36 columns x 1 row x `box_planes`; out-of-range elements read as zero
static bool make_row_map(CUtensorMap* m, const float* base, int W, int H, long planes, int box_planes) {
  EncodeTiledFn enc = encode_tiled();
  if (!enc || W % 4 != 0 || ((uintptr_t)base & 15) != 0) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
  const cuuint32_t box[3] = {36, 1, (cuuint32_t)box_planes};
  const cuuint32_t estr[3] = {1, 1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The pipelined (three-warp) form is an opt-in variant for the single-sweep case (BBD_PIPE=1 in the environment or
// -DBBD_USE_PIPE=1): parity-green on the B200, but measured slower than the one-warp streaming form (0.453 against
// 0.418 ms: its three stages are unequal, the gather warp is busy 84 % of the time, the backward warp 53 % --
// profiles/README.md), so the streaming form stays the default.
#ifndef BBD_USE_PIPE
#define BBD_USE_PIPE 0
#endif
static bool use_pipe() {
  const char* e = getenv("BBD_PIPE");  // read per launch: tests switch forms inside one process
  return e ? (e[0] != '0') : (BBD_USE_PIPE != 0);
}

template <int K, bool GRAD, bool MULTI, bool WING = false>
static int launch_stream(const bbd_reproj_args* a, cudaStream_t stream) {
  const int n_units = a->num_scales * a->batch * parts_used(a, WING);
  const int blocks = (n_units + BBD_STREAM_WARPS - 1) / BBD_STREAM_WARPS;
  const int seg_rows = (MULTI && !WING) ? BBD_STREAM_RHM : seg_rows_for(a);
  const int stride = bbd_reproj_tiles(a->height, a->width);
#if BBD_STREAM_TMA
  CUtensorMap tt, td, ti;
  if (make_row_map(&tt, a->target, a->width, a->height, 3L * a->batch, 3) &&
      make_row_map(&td, a->depth, a->width, a->height, (long)a->num_scales * a->batch, 1) &&
      make_row_map(&ti, a->ident_min, a->width, a->height, a->batch, 1)) {
    if (!MULTI && use_pipe()) {
      static bool configured_p = false;
      constexpr size_t smem_p = (size_t)PipeSmem<K, GRAD>::FLOATS * sizeof(float);
      if (!configured_p) {
        cudaError_t e = cudaFuncSetAttribute(reproj_pipe_kernel<K, GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p);
        if (e != cudaSuccess) return fail((int)e, "reproj_pipe_kernel: shared memory attribute");
        configured_p = true;
      }
      reproj_pipe_kernel<K, GRAD><<<n_units, GRAD ? 96 : 64, smem_p, stream>>>(*a, n_units, stride, tt, td, ti, seg_rows);
      return check_launch("reproj_pipe_kernel");
    }
    static bool configured = false;
    constexpr size_t smem = (size_t)BBD_STREAM_WARPS * StreamSmem<K, true, MULTI, GRAD, MULTI && !WING>::FLOATS * sizeof(float);
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(reproj_stream_tma_kernel<K, GRAD, MULTI, WING>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return fail((int)e, "reproj_stream_tma_kernel: shared memory attribute");
      configured = true;
    }
    reproj_stream_tma_kernel<K, GRAD, MULTI, WING><<<blocks, BBD_STREAM_WARPS * 32, smem, stream>>>(*a, n_units, stride, tt, td, ti, seg_rows);
    return check_launch("reproj_stream_tma_kernel");
  }
#endif
  // widths that are not a multiple of four floats (or unaligned planes) cannot be described to the TMA unit
  static bool configured = false;
  constexpr size_t smem = (size_t)BBD_STREAM_WARPS * StreamSmem<K, false, MULTI, GRAD, MULTI && !WING>::FLOATS * sizeof(float);
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(reproj_stream_kernel<K, GRAD, MULTI, WING>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "reproj_stream_kernel: shared memory attribute");
    configured = true;
  }
  reproj_stream_kernel<K, GRAD, MULTI, WING><<<blocks, BBD_STREAM_WARPS * 32, smem, stream>>>(*a, n_units, stride, seg_rows);
  return check_launch("reproj_stream_kernel");
}

extern "C" {

int bbd_version(void) { return BBD_ABI_VERSION; }
const char* bbd_last_error_string(void) { return g_err; }

int bbd_ident_forward(const bbd_ident_args* a, bbd_stream_t stream) {
  if (!a || !a->target || !a->ident_min || !a->tab.hdr || !a->tab.ident) return fail(BBD_E_ARG, "ident: null argument");
  if (a->batch <= 0 || a->height < 2 || a->width < 2) return fail(BBD_E_ARG, "ident: bad size");
  if (!a->force_tile) {
    RgbaPtrs rp;
    for (int f = 0; f < BBD_MAX_FRAMES; ++f) rp.p[f] = a->frames_rgba[f];
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int seg_rows = ident_seg_rows(a->height, a->width, a->batch, sms * 16);
    const int n_units = a->batch * IdentGeo::strips(a->width) * ((a->height + seg_rows - 1) / seg_rows);
    ident_stream_kernel<<<n_units, 32, 0, (cudaStream_t)stream>>>(*a, rp, n_units, seg_rows);
    return check_launch("ident_stream_kernel");
  }
  dim3 grid((a->width + SCfg::TW - 1) / SCfg::TW, (a->height + SCfg::TH - 1) / SCfg::TH, a->batch);
  const size_t smem = IdentStripSmem<SCfg>::floats() * sizeof(float);
  static bool configured = false;  // the attribute sticks to the function: set once, checked
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(ident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail((int)e, "ident_kernel: shared memory attribute");
    configured = true;
  }
  ident_kernel<<<grid, SCfg::NT, smem, (cudaStream_t)stream>>>(*a);
  return check_launch("ident_kernel");
}

int bbd_reproj_fused(const bbd_reproj_args* a, bbd_stream_t stream) {
  if (!a || !a->target || !a->depth || !a->inv_K || !a->P || !a->ident_min || !a->loss_part || !a->tab.hdr || !a->tab.rep)
    return fail(BBD_E_ARG, "reproj: null argument");
  if (a->need_grad && (!a->gpose_part || !a->gdepth)) return fail(BBD_E_ARG, "reproj: gradient buffers missing");
  if (a->batch <= 0 || a->height < 2 || a->width < 2 || a->num_scales <= 0) return fail(BBD_E_ARG, "reproj: bad size");
  if (a->max_rep < 1 || a->max_rep > BBD_MAX_REP) return fail(BBD_E_RANGE, "reproj: max_rep out of range");
  if (a->tickets && !bbd_reproj_finalizes_itself(a)) return fail(BBD_E_ARG, "reproj: tickets given but pair_sum / loss_out / gpose_out missing or tile kernel selected");
  if (use_stream(a)) {
    cudaStream_t st = (cudaStream_t)stream;
    if (a->max_rep == 1) return a->need_grad ? launch_stream<1, true, false>(a, st) : launch_stream<1, false, false>(a, st);
    if (a->max_rep == 2) return a->need_grad ? launch_stream<2, true, false>(a, st) : launch_stream<2, false, false>(a, st);
#if !BBD_STREAM_ASYNC
    if (split_multi(a)) {  // selection round, then the gradient round reading a->winner
      if (int rc = launch_stream<2, false, true>(a, st)) return rc;
      return launch_stream<2, true, true, true>(a, st);
    }
    return a->need_grad ? launch_stream<2, true, true>(a, st) : launch_stream<2, false, true>(a, st);
#endif
  }
  // keep every candidate's warped tile resident while that still allows three blocks per SM
  const bool keep = StripSmem<SCfg>::floats(a->max_rep) * sizeof(float) <= 75 * 1024;
  const size_t smem = StripSmem<SCfg>::floats(keep ? a->max_rep : 1) * sizeof(float);
  if (smem > 227 * 1024) return fail(BBD_E_RANGE, "reproj: shared memory budget exceeded");
  dim3 grid((a->width + SCfg::TW - 1) / SCfg::TW, (a->height + SCfg::TH - 1) / SCfg::TH, a->num_scales * a->batch);
  static size_t configured[4] = {0, 0, 0, 0};  // largest dynamic shared-memory size granted per variant
  int rc = 0;
  auto launch = [&](auto kern, int which) {
    if (configured[which] < smem) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) { rc = fail((int)e, "reproj_kernel: shared memory attribute"); return; }
      configured[which] = smem;
    }
    kern<<<grid, SCfg::NT, smem, (cudaStream_t)stream>>>(*a);
  };
  if (a->need_grad) {
    if (keep) launch(reproj_kernel<true, true>, 0); else launch(reproj_kernel<true, false>, 1);
  } else {
    if (keep) launch(reproj_kernel<false, true>, 2); else launch(reproj_kernel<false, false>, 3);
  }
  if (rc) return rc;
  return check_launch("reproj_kernel");
}

int bbd_reproj_finalizes_itself(const bbd_reproj_args* a) {
  return a && use_stream(a) && a->max_rep <= 2 && a->tickets && a->pair_sum && a->loss_out && (!a->need_grad || a->gpose_out) ? 1 : 0;
}

const char* bbd_reproj_kernel_name(const bbd_reproj_args* a) {
  if (!a) return "";
  if (use_stream(a)) {
    const bool tma = BBD_STREAM_TMA && encode_tiled() && a->width % 4 == 0 && !(((uintptr_t)a->target | (uintptr_t)a->depth | (uintptr_t)a->ident_min) & 15);
    static char name[64];
    if (tma && a->max_rep <= 2 && use_pipe())
      snprintf(name, sizeof(name), "bbd::reproj_pipe_kernel<%d, %d>", a->max_rep == 1 ? 1 : 2, a->need_grad ? 1 : 0);
    else
      if (split_multi(a))  // selection launch <2, 0, 1> followed by the gradient launch named here
        snprintf(name, sizeof(name), "bbd::reproj_stream%s_kernel<2, 1, 1, 1>", tma ? "_tma" : "");
      else
        snprintf(name, sizeof(name), "bbd::reproj_stream%s_kernel<%d, %d, %d>", tma ? "_tma" : "", a->max_rep == 1 ? 1 : 2, a->need_grad ? 1 : 0,
                 a->max_rep > 2 ? 1 : 0);
    return name;
  }
  const bool keep = StripSmem<SCfg>::floats(a->max_rep) * sizeof(float) <= 75 * 1024;
  if (a->need_grad) return keep ? "bbd::reproj_kernel<1, 1>" : "bbd::reproj_kernel<1, 0>";
  return keep ? "bbd::reproj_kernel<0, 1>" : "bbd::reproj_kernel<0, 0>";
}

int bbd_reproj_finalize(const bbd_reproj_args* a, float* loss, float* gpose, bbd_stream_t stream) {
  if (!a || !loss || !a->loss_part) return fail(BBD_E_ARG, "finalize: null argument");
  if (gpose && !a->gpose_part) return fail(BBD_E_ARG, "finalize: no pose partials");
  const int ntiles = bbd_reproj_tiles(a->height, a->width);
  const int blocks = a->num_scales * (1 + (gpose ? a->num_pose : 0));
  reproj_finalize_kernel<<<blocks, FIN_NT, 0, (cudaStream_t)stream>>>(*a, loss, gpose, ntiles, parts_used(a, false), parts_used(a, true));
  return check_launch("reproj_finalize_kernel");
}

static int smooth_max_parts(int levels, const int32_t* h, const int32_t* w) {
  int mc = 1;
  for (int l = 0; l < levels; ++l) mc = std::max(mc, std::max(sm_chunks(h[l], w[l]), smr_blocks(h[l], w[l])));
  return mc;
}
// partial-sum slots (levels,B,4,parts) + the per-sample scalars (levels,B,2) + the ticket of the last-block reduction
size_t bbd_smooth_scratch_floats(int32_t batch, int32_t levels, const int32_t* h, const int32_t* w) {
  return (size_t)levels * batch * 4 * smooth_max_parts(levels, h, w) + (size_t)levels * batch * 2 + 4;
}

int bbd_smooth_fused(const bbd_smooth_args* in, bbd_stream_t stream) {
  if (!in || !in->scratch || !in->loss) return fail(BBD_E_ARG, "smooth: null argument");
  if (in->levels < 1 || in->levels > BBD_MAX_SCALES || in->batch <= 0 || in->batch > 256) return fail(BBD_E_RANGE, "smooth: bad level count / batch");
  if (in->defer_norm && !in->coef) return fail(BBD_E_ARG, "smooth: defer_norm needs coef");
  bbd_smooth_args a = *in;
  int nbx = 1, nby = 1;
  unsigned total = 0;
  for (int l = 0; l < a.levels; ++l) {
    if (!a.disp[l] || !a.img[l] || a.h[l] < 2 || a.w[l] < 2) return fail(BBD_E_ARG, "smooth: bad level");
    nbx = std::max(nbx, smr_nbx(a.w[l]));
    nby = std::max(nby, smr_nby(a.h[l]));
    total += (unsigned)(a.batch * smr_blocks(a.h[l], a.w[l]));
  }
  const int mc = smooth_max_parts(a.levels, a.h, a.w);
  a.max_chunks = mc;
  float* tail = a.scratch + (size_t)a.levels * a.batch * 4 * mc;
  float* coef = a.defer_norm ? a.coef : tail;
  unsigned* ticket = reinterpret_cast<unsigned*>(tail + (size_t)a.levels * a.batch * 2);
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(ticket, 0, sizeof(unsigned), st);
  dim3 grid(nbx, nby, a.levels * a.batch);
  smooth_rows_kernel<<<grid, SMR_WARPS * 32, 0, st>>>(a, coef, ticket, total);
  if (!a.defer_norm && a.normalize) {
    bool any = false;
    for (int l = 0; l < a.levels; ++l) any = any || a.gdisp[l];
    if (any) {
      dim3 grid3(8, a.batch, a.levels);
      smooth_apply_kernel<<<grid3, 256, 0, st>>>(a, coef);
    }
  }
  return check_launch("smooth kernels");
}

int bbd_disp_to_depth_forward(const bbd_d2d_args* a, bbd_stream_t stream) {
  if (!a || !a->depth) return fail(BBD_E_ARG, "d2d forward: null argument");
  if (a->levels < 1 || a->levels > BBD_MAX_SCALES) return fail(BBD_E_RANGE, "d2d: bad level count");
  for (int l = 0; l < a->levels; ++l)
    if (!a->disp[l] || a->h[l] < 1 || a->w[l] < 1) return fail(BBD_E_ARG, "d2d forward: bad level");
  const size_t rows = (size_t)a->batch * a->height;
  dim3 grid((unsigned)(((a->width + 3) / 4 + 127) / 128), (unsigned)std::min<size_t>(rows, kRowBlocks), a->levels);
  d2d_forward_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(*a);
  return check_launch("d2d_forward_kernel");
}

static int d2d_backward_check(const bbd_d2d_args* a) {
  if (!a || !a->depth || !a->gdepth || !a->gscale) return fail(BBD_E_ARG, "d2d backward: null argument");
  if (a->levels < 1 || a->levels > BBD_MAX_SCALES) return fail(BBD_E_RANGE, "d2d: bad level count");
  for (int l = 0; l < a->levels; ++l) {
    if (!a->gdisp[l]) return fail(BBD_E_ARG, "d2d backward: bad level");
    if (a->height % a->h[l] || a->width % a->w[l] || a->height / a->h[l] > 8 || a->width / a->w[l] > 8)
      return fail(BBD_E_RANGE, "d2d backward: scale factor must be an integer <= 8");
  }
  return 0;
}

int bbd_disp_to_depth_backward_pass1(const bbd_d2d_args* a, bbd_stream_t stream) {
  if (int rc = d2d_backward_check(a)) return rc;
  if (!a->scratch) return 0;
  int wsep = 0;
  for (int l = 0; l < a->levels; ++l)
    if (d2d_sep_factor(*a, l)) wsep = std::max(wsep, a->w[l]);
  if (!wsep) return 0;
  const size_t rows = (size_t)a->batch * a->height;
  dim3 hgrid((unsigned)((wsep + 127) / 128), (unsigned)std::min<size_t>(rows, kRowBlocks), a->levels);
  d2d_hpass_kernel<<<hgrid, 128, 0, (cudaStream_t)stream>>>(*a);
  return check_launch("d2d_hpass_kernel");
}

int bbd_disp_to_depth_backward_pass2(const bbd_d2d_args* a, int32_t level_begin, int32_t level_end, bbd_stream_t stream) {
  if (int rc = d2d_backward_check(a)) return rc;
  if (level_begin < 0 || level_end > a->levels || level_begin > level_end) return fail(BBD_E_RANGE, "d2d backward: bad level range");
  if (level_begin == level_end) return 0;
  int wmax = 1, hmax = 1;
  for (int l = level_begin; l < level_end; ++l) {
    wmax = std::max(wmax, a->w[l]);
    hmax = std::max(hmax, a->h[l]);
  }
  const size_t rows = (size_t)a->batch * hmax;
  dim3 grid((unsigned)((wmax + 127) / 128), (unsigned)std::min<size_t>(rows, kRowBlocks), level_end - level_begin);
  d2d_backward_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(*a, level_begin);
  return check_launch("d2d_backward_kernel");
}

int bbd_disp_to_depth_backward(const bbd_d2d_args* a, bbd_stream_t stream) {
  if (int rc = d2d_backward_check(a)) return rc;
  bool fused = (((uintptr_t)a->gdepth | (uintptr_t)a->depth) & 15) == 0 && 2 * (size_t)a->width * sizeof(float) <= 48 * 1024;
  int max_h = 1;
  for (int l = 0; l < a->levels; ++l) {
    fused = fused && d2d_fused_factor(*a, l) != 0;
    max_h = std::max(max_h, a->h[l]);
  }
  if (fused) {  // every level in one launch, no scratch plane
    D2DRowList list;
    int order[BBD_MAX_SCALES];
    for (int l = 0; l < a->levels; ++l) order[l] = l;
    std::sort(order, order + a->levels, [&](int x, int y) { return a->h[x] < a->h[y]; });  // coarsest (most rows read per row) first
    list.begin[0] = 0;
    for (int j = 0; j < a->levels; ++j) {
      list.level[j] = order[j];
      list.begin[j + 1] = list.begin[j] + a->batch * a->h[order[j]];
    }
    for (int j = a->levels; j < BBD_MAX_SCALES; ++j) { list.level[j] = 0; list.begin[j + 1] = list.begin[a->levels]; }
    const int threads = std::min(256, std::max(32, ((a->width / 4 + 31) / 32) * 32));
    static int per_sm = 0;  // resident blocks per SM of this kernel at this block size (queried once)
    static int per_sm_threads = 0;
    if (per_sm_threads != threads) {
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, d2d_backward_fused_kernel, threads, 2 * (size_t)a->width * sizeof(float)) != cudaSuccess || per_sm < 1) per_sm = 1;
      per_sm_threads = threads;
    }
    int sms = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = std::min(list.begin[a->levels], sms * per_sm);
    d2d_backward_fused_kernel<<<blocks, threads, 2 * (size_t)a->width * sizeof(float), (cudaStream_t)stream>>>(*a, list);
    return check_launch("d2d_backward_fused_kernel");
  }
  if (int rc = bbd_disp_to_depth_backward_pass1(a, stream)) return rc;
  return bbd_disp_to_depth_backward_pass2(a, 0, a->levels, stream);
}

size_t bbd_d2d_scratch_floats(const bbd_d2d_args* a) {
  if (!a) return 0;
  return d2d_scratch_offset(*a, a->levels);
}

int bbd_pose_forward(int32_t n, const float* axisangle, const float* translation, int32_t invert, float* T,
                     bbd_stream_t stream) {
  if (!axisangle || !translation || !T) return fail(BBD_E_ARG, "pose: null argument");
  if (n <= 0) return 0;
  pose_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(n, axisangle, translation, invert, T);
  return check_launch("pose_kernel");
}

int bbd_pose_backward(int32_t n, const float* axisangle, const float* translation, int32_t invert, const float* gT,
                      float* gaxisangle, float* gtranslation, bbd_stream_t stream) {
  if (!axisangle || !translation || !gT || !gaxisangle || !gtranslation) return fail(BBD_E_ARG, "pose backward: null argument");
  if (n <= 0) return 0;
  pose_grad_kernel<<<(n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(n, axisangle, translation, invert, gT, gaxisangle,
                                                                  gtranslation);
  return check_launch("pose_grad_kernel");
}

int bbd_pose_pack_forward(int32_t n_pose, const float* K, const int32_t* k_row, const float* T, float* P,
                          bbd_stream_t stream) {
  if (!K || !k_row || !T || !P) return fail(BBD_E_ARG, "pose_pack: null argument");
  if (n_pose <= 0) return 0;
  pose_pack_kernel<<<(n_pose * 12 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n_pose, K, k_row, T, P);
  return check_launch("pose_pack_kernel");
}

int bbd_pose_pack_backward(int32_t n_pose, const float* K, const int32_t* k_row, const float* gP, float* gT,
                           bbd_stream_t stream) {
  if (!K || !k_row || !gP || !gT) return fail(BBD_E_ARG, "pose_pack backward: null argument");
  if (n_pose <= 0) return 0;
  pose_pack_grad_kernel<<<(n_pose * 16 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(n_pose, K, k_row, gP, gT);
  return check_launch("pose_pack_grad_kernel");
}

int bbd_warp_forward(int32_t n, int32_t height, int32_t width, const float* images, const float* depth, const float* inv_K,
                     const float* P, float* warped, float* grid, bbd_stream_t stream) {
  if (!images || !depth || !inv_K || !P || !warped) return fail(BBD_E_ARG, "warp: null argument");
  if (n == 0) return 0;
  warp_kernel<<<grid_for((size_t)n * height * width, 256), 256, 0, (cudaStream_t)stream>>>(n, height, width, images, depth,
                                                                                         inv_K, P, warped, grid);
  return check_launch("warp_kernel");
}

int bbd_backproject_forward(int32_t n, int32_t height, int32_t width, const float* depth, const float* inv_K, float* points,
                            bbd_stream_t stream) {
  if (!depth || !inv_K || !points) return fail(BBD_E_ARG, "backproject: null argument");
  if (n == 0) return 0;
  backproject_kernel<<<grid_for((size_t)n * height * width, 256), 256, 0, (cudaStream_t)stream>>>(n, height, width, depth,
                                                                                                inv_K, points);
  return check_launch("backproject_kernel");
}

int bbd_backproject_backward(int32_t n, int32_t height, int32_t width, const float* inv_K, const float* gpoints,
                             float* gdepth, bbd_stream_t stream) {
  if (!inv_K || !gpoints || !gdepth) return fail(BBD_E_ARG, "backproject backward: null argument");
  if (n == 0) return 0;
  backproject_grad_kernel<<<grid_for((size_t)n * height * width, 256), 256, 0, (cudaStream_t)stream>>>(
      n, height, width, inv_K, gpoints, gdepth);
  return check_launch("backproject_grad_kernel");
}

int bbd_project_forward(int32_t n, int32_t height, int32_t width, const float* points, const float* P, float eps,
                        float* pix, bbd_stream_t stream) {
  if (!points || !P || !pix) return fail(BBD_E_ARG, "project: null argument");
  if (n == 0) return 0;
  project_kernel<<<grid_for((size_t)n * height * width, 256), 256, 0, (cudaStream_t)stream>>>(n, height, width, points, P,
                                                                                            eps, pix);
  return check_launch("project_kernel");
}

int bbd_project_chunks(int32_t height, int32_t width) { return (height * width + PJ_CHUNK - 1) / PJ_CHUNK; }

int bbd_project_backward(int32_t n, int32_t height, int32_t width, const float* points, const float* P, float eps,
                         const float* gpix, float* gpoints, float* gP_part, bbd_stream_t stream) {
  if (!points || !P || !gpix || !gpoints || !gP_part) return fail(BBD_E_ARG, "project backward: null argument");
  if (n == 0) return 0;
  dim3 grid(bbd_project_chunks(height, width), n);
  project_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(n, height, width, points, P, eps, gpix, gpoints, gP_part);
  return check_launch("project_grad_kernel");
}

int bbd_grid_sample_forward(int32_t n, int32_t channels, int32_t height, int32_t width, int32_t out_h, int32_t out_w,
                            const float* images, const float* grid, float* out, bbd_stream_t stream) {
  if (!images || !grid || !out) return fail(BBD_E_ARG, "grid_sample: null argument");
  if (n * channels == 0 || out_h * out_w == 0) return 0;
  grid_sample_kernel<<<grid_for((size_t)n * out_h * out_w, 256), 256, 0, (cudaStream_t)stream>>>(
      n, channels, height, width, out_h * out_w, images, grid, out);
  return check_launch("grid_sample_kernel");
}

int bbd_grid_sample_backward(int32_t n, int32_t channels, int32_t height, int32_t width, int32_t out_h, int32_t out_w,
                             const float* images, const float* grid, const float* gout, float* ggrid,
                             bbd_stream_t stream) {
  if (!images || !grid || !gout || !ggrid) return fail(BBD_E_ARG, "grid_sample backward: null argument");
  if (n == 0 || out_h * out_w == 0) return 0;
  grid_sample_grad_kernel<<<grid_for((size_t)n * out_h * out_w, 256), 256, 0, (cudaStream_t)stream>>>(
      n, channels, height, width, out_h * out_w, images, grid, gout, ggrid);
  return check_launch("grid_sample_grad_kernel");
}

int bbd_loss_combine_forward(int32_t n, const float* reproj, const float* smooth, const float* weight, float num_scales,
                             float* per_scale, float* total, bbd_stream_t stream) {
  if (!reproj || !smooth || !weight || !per_scale || !total) return fail(BBD_E_ARG, "loss_combine: null argument");
  if (n < 1 || n > BBD_MAX_SCALES || !(num_scales > 0.0f)) return fail(BBD_E_RANGE, "loss_combine: bad term count");
  loss_combine_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(n, reproj, smooth, weight, num_scales, per_scale, total);
  return check_launch("loss_combine_kernel");
}

int bbd_loss_combine_backward(int32_t n, const float* g_total, const float* g_per_scale, const float* weight,
                              float num_scales, float* g_reproj, float* g_smooth, bbd_stream_t stream) {
  if (!weight || !g_reproj || !g_smooth) return fail(BBD_E_ARG, "loss_combine backward: null argument");
  if (n < 1 || n > BBD_MAX_SCALES || !(num_scales > 0.0f)) return fail(BBD_E_RANGE, "loss_combine: bad term count");
  loss_combine_grad_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(n, g_total, g_per_scale, weight, num_scales, g_reproj, g_smooth);
  return check_launch("loss_combine_grad_kernel");
}

int bbd_project_coords(int32_t n, int32_t height, int32_t width, const float* depth, const float* inv_K, const float* P,
                       float* grid, float* pix, bbd_stream_t stream) {
  if (!depth || !inv_K || !P || (!grid && !pix)) return fail(BBD_E_ARG, "project_coords: null argument");
  if (n <= 0) return 0;
  stream_coords_kernel<<<grid_for((size_t)n * height * width, 256), 256, 0, (cudaStream_t)stream>>>(n, height, width, depth, inv_K,
                                                                                                   P, grid, pix);
  return check_launch("stream_coords_kernel");
}

int bbd_pack_rgba(int32_t n, int32_t height, int32_t width, const float* planar, float* rgba, bbd_stream_t stream) {
  if (!planar || !rgba) return fail(BBD_E_ARG, "pack_rgba: null argument");
  if (n <= 0) return 0;
  const int HW = height * width;
  const bool vec = (HW % 4 == 0) && ((uintptr_t)planar % 16 == 0) && ((uintptr_t)rgba % 16 == 0);
  if (vec)
    pack_rgba_kernel<<<grid_for((size_t)n * HW / 4, 256), 256, 0, (cudaStream_t)stream>>>(n, HW, planar, reinterpret_cast<float4*>(rgba));
  else
    pack_rgba_scalar_kernel<<<grid_for((size_t)n * HW, 256), 256, 0, (cudaStream_t)stream>>>(n, HW, planar, reinterpret_cast<float4*>(rgba));
  return check_launch("pack_rgba_kernel");
}

int bbd_u8_to_f32(const uint8_t* src, float* dst, size_t n, bbd_stream_t stream) {
  if (!src || !dst) return fail(BBD_E_ARG, "u8_to_f32: null argument");
  if (n == 0) return 0;
  const bool aligned = ((uintptr_t)src % 16 == 0) && ((uintptr_t)dst % 16 == 0);
  const size_t n16 = aligned ? n / 16 : 0;
  if (n16)
    u8_to_f32_kernel<<<grid_for(n16, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint4*>(src),
                                                                            reinterpret_cast<float4*>(dst), n16);
  const size_t done = n16 * 16;
  if (done < n)
    u8_to_f32_tail_kernel<<<(unsigned)((n - done + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, dst, done, n);
  return check_launch("u8_to_f32_kernel");
}

int bbd_grid_sample_dest_keys(int32_t n, int32_t height, int32_t width, int32_t out_h, int32_t out_w, const float* grid,
                              int32_t* keys, bbd_stream_t stream) {
  if (!grid || !keys) return fail(BBD_E_ARG, "grid_sample keys: null argument");
  if (n <= 0) return 0;
  if ((size_t)n * height * width >= (size_t)1 << 31 || (size_t)n * out_h * out_w >= (size_t)1 << 31)
    return fail(BBD_E_RANGE, "grid_sample keys: more than 2^31 elements");
  gs_dest_keys_kernel<<<grid_for((size_t)n * out_h * out_w, 256), 256, 0, (cudaStream_t)stream>>>(n, height, width, out_h * out_w, grid, keys);
  return check_launch("gs_dest_keys_kernel");
}

int bbd_grid_sample_backward_image(int32_t n, int32_t channels, int32_t height, int32_t width, int32_t out_h, int32_t out_w,
                                   const float* grid, const float* gout, const int32_t* keys_sorted, const int32_t* order,
                                   int32_t* seg_start, float* gimages, bbd_stream_t stream) {
  if (!grid || !gout || !keys_sorted || !order || !seg_start || !gimages) return fail(BBD_E_ARG, "grid_sample image gradient: null argument");
  if (n <= 0) return 0;
  const int n_items = n * out_h * out_w, n_keys = n * height * width;
  gs_segment_kernel<<<grid_for((size_t)n_items + 1, 256), 256, 0, (cudaStream_t)stream>>>(keys_sorted, n_items, n_keys, seg_start);
  gs_image_grad_kernel<<<grid_for((size_t)n * channels * height * width, 256), 256, 0, (cudaStream_t)stream>>>(
      n, channels, height, width, out_h * out_w, grid, gout, seg_start, order, gimages);
  return check_launch("gs_image_grad_kernel");
}

int bbd_ssim_forward(int32_t n, int32_t channels, int32_t height, int32_t width, const float* x, const float* y, float* out,
                     bbd_stream_t stream) {
  if (!x || !y || !out) return fail(BBD_E_ARG, "ssim: null argument");
  if (height < 2 || width < 2) return fail(BBD_E_RANGE, "ssim: reflection padding needs at least 2 pixels");
  if (n * channels == 0) return 0;
  ssim_kernel<<<grid_for((size_t)n * channels * height * width, 256), 256, 0, (cudaStream_t)stream>>>(n * channels, height,
                                                                                                    width, x, y, out);
  return check_launch("ssim_kernel");
}

int bbd_ssim_backward(int32_t n, int32_t channels, int32_t height, int32_t width, const float* x, const float* y,
                      const float* gout, float* gx, float* gy, bbd_stream_t stream) {
  if (!x || !y || !gout) return fail(BBD_E_ARG, "ssim backward: null argument");
  if (n * channels == 0 || (!gx && !gy)) return 0;
  ssim_grad_kernel<<<grid_for((size_t)n * channels * height * width, 128), 128, 0, (cudaStream_t)stream>>>(
      n * channels, height, width, x, y, gout, gx, gy);
  return check_launch("ssim_grad_kernel");
}

// what both frame-gradient calls read; sizes and index ranges
static int frame_grad_check(const bbd_reproj_args* a, const bbd_frame_grad_args* f, const char* who) {
  static thread_local char msg[128];
  if (!a || !f || !a->target || !a->depth || !a->inv_K || !a->P || !a->tab.hdr || !a->tab.rep || !a->tab.ident ||
      !f->gpred || !f->gident) {
    snprintf(msg, sizeof(msg), "%s: null argument", who);
    return fail(BBD_E_ARG, msg);
  }
  if (a->batch <= 0 || a->height < 2 || a->width < 2 || a->num_scales <= 0) {
    snprintf(msg, sizeof(msg), "%s: bad size", who);
    return fail(BBD_E_ARG, msg);
  }
  size_t rows = 0;
  for (int s = 0; s < BBD_MAX_FRAMES; ++s) {
    if (f->stack_rows[s] < 0) {
      snprintf(msg, sizeof(msg), "%s: negative stack_rows", who);
      return fail(BBD_E_RANGE, msg);
    }
    rows += (size_t)f->stack_rows[s];
  }
  const size_t HW = (size_t)a->height * a->width;
  if (a->num_scales > BBD_MAX_SCALES || a->max_rep < 1 || a->max_rep > BBD_MAX_REP ||
      (size_t)a->num_scales * a->batch * a->max_rep * HW >= ((size_t)1 << 31) || rows * HW >= ((size_t)1 << 31) - 1) {
    snprintf(msg, sizeof(msg), "%s: scales / max_rep / entry count out of range", who);
    return fail(BBD_E_RANGE, msg);
  }
  return 0;
}

int bbd_frame_grad(const bbd_reproj_args* a, const bbd_frame_grad_args* f, bbd_stream_t stream) {
  if (int e = frame_grad_check(a, f, "frame_grad")) return e;
  if (!a->winner || !f->gscale || !f->keys || (!a->no_ssim && !f->coef))
    return fail(BBD_E_ARG, "frame_grad: winner / gscale / keys / coef missing");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t HW = (size_t)a->height * a->width;
  if (!a->no_ssim)
    frame_grad_coef_kernel<<<grid_for((size_t)a->num_scales * a->batch * HW, 256), 256, 0, st>>>(*a, *f);
  frame_grad_pred_kernel<<<grid_for((size_t)a->batch * HW, 256), 256, 0, st>>>(*a, *f);
  return check_launch("frame_grad kernels");
}

int bbd_frame_grad_stacks(const bbd_reproj_args* a, const bbd_frame_grad_args* f, bbd_stream_t stream) {
  if (int e = frame_grad_check(a, f, "frame_grad_stacks")) return e;
  if (!f->keys_sorted || !f->order || !f->seg_start) return fail(BBD_E_ARG, "frame_grad_stacks: sorted keys / order / seg_start missing");
  int rows = 0;
  for (int s = 0; s < BBD_MAX_FRAMES; ++s) rows += f->stack_rows[s];
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t HW = (size_t)a->height * a->width;
  const int n_items = (int)((size_t)a->num_scales * a->batch * a->max_rep * HW), n_keys = (int)(rows * HW);
  gs_segment_kernel<<<grid_for((size_t)n_items + 1, 256), 256, 0, st>>>(f->keys_sorted, n_items, n_keys, f->seg_start);
  frame_grad_stack_kernel<<<grid_for((size_t)rows * 3 * HW, 256), 256, 0, st>>>(*a, *f, rows);
  return check_launch("frame_grad_stack_kernel");
}

int bbd_smooth_image_grad(const bbd_smooth_img_args* a, bbd_stream_t stream) {
  if (!a || !a->gscale) return fail(BBD_E_ARG, "smooth image gradient: null argument");
  if (a->levels < 1 || a->levels > BBD_MAX_SCALES || a->batch <= 0 || a->batch > 65535)
    return fail(BBD_E_RANGE, "smooth image gradient: bad level count / batch");
  int mx = 1;
  for (int l = 0; l < a->levels; ++l) {
    if (!a->gimg[l]) continue;
    if (!a->disp[l] || !a->img[l] || a->h[l] < 2 || a->w[l] < 2) return fail(BBD_E_ARG, "smooth image gradient: bad level");
    mx = std::max(mx, a->h[l] * a->w[l]);
  }
  dim3 grid(std::min((mx + 255) / 256, 64), a->batch, a->levels);
  smooth_image_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*a);
  return check_launch("smooth_image_grad_kernel");
}

}  // extern "C"
