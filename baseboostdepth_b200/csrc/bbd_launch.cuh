// Launch decisions of the loss kernels: which kernel instance serves a call and how the call is cut into units.
//
// Pure host functions of an ABI argument block and the device facts the caller supplies (LaunchDevice).  The
// library (bbd_kernels.cu) launches what they describe; the CPU harness (tests/emu) steps the same list of
// launches, so a launch rule is written once.  No CUDA API call here: compiles under nvcc and g++ alike.
#pragma once
#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

#include "bbd_ops.cuh"
#include "bbd_smooth.cuh"
#include "bbd_strip.cuh"
#include "bbd_stream.cuh"

// Identity pre-pass and fused loss share one tile geometry: 28x16 target pixels per block of 6
// warps, lanes = columns (bbd_strip.cuh).  With two warped candidates a block needs 64 KB of shared
// memory -> 3 blocks (18 warps) per SM at 96 registers per thread.  Fewer, fatter warps beat 8 warps
// at 80 registers: the kernel gains from instruction-level parallelism inside a warp (four rows of
// gathers in flight in the warp phase, two rows walked together in the backward), not from more
// resident warps (profiles/README.md lists the measured variants).
#ifndef BBD_TILE_H
#define BBD_TILE_H 16
#endif
#ifndef BBD_WARPS
#define BBD_WARPS 6
#endif
#ifndef BBD_STREAM_MINB
#define BBD_STREAM_MINB 8  // resident warps per SM of the one-warp streaming form (224-243 registers per thread)
#endif
#ifndef BBD_STREAM_TMA
#define BBD_STREAM_TMA 1
#endif
// The pipelined (three-warp) form is an opt-in variant for the single-sweep case (BBD_PIPE=1 in the environment or
// -DBBD_USE_PIPE=1): parity-green on the B200, but measured slower than the one-warp streaming form (0.453 against
// 0.418 ms: its three stages are unequal, the gather warp is busy 84 % of the time, the backward warp 53 % --
// profiles/README.md), so the streaming form stays the default.
#ifndef BBD_USE_PIPE
#define BBD_USE_PIPE 0
#endif

namespace bbd {

using SCfg = StripCfg<BBD_TILE_H, BBD_WARPS>;

// What the caller knows about the device.
struct LaunchDevice {
  int sms;    // multiprocessors
  bool tma;   // a tensor-map encoder is available
  bool pipe;  // the pipelined form is asked for
};

inline bool pipe_requested() {
  const char* e = getenv("BBD_PIPE");  // read per launch: tests switch forms inside one process
  return e ? (e[0] != '0') : (BBD_USE_PIPE != 0);
}

// ---- alignment of caller-supplied buffers --------------------------------------------------------
// A 16-byte access (float4 / LDG.128 / STG.128, a TMA box) to a buffer the caller owns is issued only where the
// buffer's address allows it; every such access is decided here.
inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// The channel-interleaved frame copies (frames_rgba) are written and read one 16-byte pixel at a time, in every
// form: bbd_pack_rgba, bbd_ident_forward and bbd_reproj_fused reject a non-NULL entry that is not 16-byte aligned.
template <class T>
inline bool rgba_aligned(T* const* rgba) {
  for (int f = 0; f < BBD_MAX_FRAMES; ++f)
    if (!aligned16(rgba[f])) return false;
  return true;
}

// disp_to_depth forward: a thread stores its four pixels as one float4 when rows are whole float4s and the depth
// planes start on a 16-byte boundary; otherwise four scalar stores.
inline bool d2d_forward_vec(const bbd_d2d_args& a) { return a.width % 4 == 0 && aligned16(a.depth); }

// ---- fused reprojection loss ------------------------------------------------------------------
enum ReprojForm { REPROJ_TILE, REPROJ_STREAM, REPROJ_PIPE };

// One launch: reproj_stream[_tma]_kernel<K, GRAD, MULTI, WING> or reproj_pipe_kernel<K, GRAD> with `units` warps
// (pipelined: blocks) walking segments of `seg_rows` rows; reproj_kernel<GRAD, KEEP> with one block per tile.
struct KernelLaunch {
  bool grad, multi, wing;
  int units, seg_rows;
};

struct ReprojLaunch {
  ReprojForm form;
  bool keep;             // tile form: every candidate's warped tile stays in shared memory
  size_t tile_smem;      // tile form: dynamic shared memory (bytes)
  bool tma;              // streaming forms: the regular planes are staged by the TMA unit
  int k;                 // streaming forms: candidates per sweep (1 or 2)
  int n_launches;        // 1, or 2 for the selection and gradient rounds of the many-candidate form
  KernelLaunch launch[2];
  int stride;            // slots of loss_part / gpose_part per (scale, sample)
  int used, used_grad;   // slots the loss and the gradient launches fill per (scale, sample)
  bool finalizes_itself; // the streaming kernel reduces its own partials: no bbd_reproj_finalize
};

inline int tile_parts(int height, int width) {
  return ((width + SCfg::TW - 1) / SCfg::TW) * ((height + SCfg::TH - 1) / SCfg::TH);
}
// slots per (scale, sample) in loss_part / gpose_part: enough for either kernel
inline int reproj_slots(int height, int width) {
  const int a = tile_parts(height, width), b = StreamGeo::strips(width) * stream_max_segs(height),
            c = StreamGeoM::units(height, width);
  return a > b ? (a > c ? a : c) : (b > c ? b : c);
}

inline bool reproj_uses_stream(const bbd_reproj_args& a) {
  if (a.force_tile || a.min_rep < 1 || a.max_rep > BBD_MAX_REP) return false;
  bool any = false;
  for (int f = 0; f < BBD_MAX_FRAMES; ++f) {
    if (a.frames[f] && !a.frames_rgba[f]) return false;
    any = any || a.frames_rgba[f];
  }
  return any;
}

inline ReprojLaunch reproj_launch(const bbd_reproj_args& a, const LaunchDevice& dev) {
  ReprojLaunch L = {};
  L.stride = reproj_slots(a.height, a.width);
  const int pairs = a.num_scales * a.batch;
  if (!reproj_uses_stream(a)) {
    // one block per tile of one (scale, sample); keep every candidate's warped tile resident while that still
    // allows three blocks per SM
    L.form = REPROJ_TILE;
    L.keep = StripSmem<SCfg>::floats(a.max_rep) * sizeof(float) <= 75 * 1024;
    L.tile_smem = StripSmem<SCfg>::floats(L.keep ? a.max_rep : 1) * sizeof(float);
    L.used = L.used_grad = tile_parts(a.height, a.width);
    L.n_launches = 1;
    L.launch[0] = {a.need_grad != 0, false, false, pairs * L.used, SCfg::TH};
    return L;
  }
  // widths that are not a multiple of four floats (or unaligned planes) cannot be described to the TMA unit
  L.tma = BBD_STREAM_TMA && dev.tma && a.width % 4 == 0 && aligned16(a.target) && aligned16(a.depth) && aligned16(a.ident_min);
  L.k = a.max_rep == 1 ? 1 : 2;
  const bool multi = a.max_rep > 2;
  L.form = L.tma && !multi && dev.pipe ? REPROJ_PIPE : REPROJ_STREAM;
  const int slots = dev.sms * BBD_STREAM_MINB;
  // single-sweep segments: as tall as fills the resident warps in the fewest rounds
  const int rh = multi ? stream_seg_rows_uneven(a.height, a.width, pairs, slots) : stream_seg_rows(a.height, a.width, pairs, slots);
  const int sweep_parts = StreamGeo::strips(a.width) * ((a.height + rh - 1) / rh);
  const KernelLaunch single = {a.need_grad != 0, false, false, pairs * sweep_parts, rh};
  // many candidates: short segments carrying the selection plane in shared memory
  const KernelLaunch select = {a.need_grad != 0, true, false, pairs * StreamGeoM::units(a.height, a.width), BBD_STREAM_RHM};
  if (!multi) {
    L.n_launches = 1;
    L.launch[0] = single;
    L.used = L.used_grad = sweep_parts;
  } else if (a.need_grad && a.winner) {
    // with the winner plane the gradients run as two launches: a forward-only selection launch (twelve warps per
    // SM) and a gradient launch that reads the winners (tall segments)
    L.n_launches = 2;
    L.launch[0] = select;
    L.launch[0].grad = false;
    L.launch[1] = single;
    L.launch[1].multi = L.launch[1].wing = true;
    L.used = StreamGeoM::units(a.height, a.width);
    L.used_grad = sweep_parts;
  } else {
    L.n_launches = 1;
    L.launch[0] = select;
    L.used = L.used_grad = StreamGeoM::units(a.height, a.width);
  }
  L.finalizes_itself = !multi && a.tickets && a.pair_sum && a.loss_out && (!a.need_grad || a.gpose_out);
  return L;
}

// Calls f(k, grad, multi, wing) with std::integral_constant arguments naming the kernel instance of launch l.
template <class F>
auto with_stream_instance(const ReprojLaunch& L, const KernelLaunch& l, F&& f) {
  typedef std::true_type T;
  typedef std::false_type N;
  typedef std::integral_constant<int, 1> K1;
  typedef std::integral_constant<int, 2> K2;
  if (L.k == 1) return l.grad ? f(K1(), T(), N(), N()) : f(K1(), N(), N(), N());
  if (!l.multi) return l.grad ? f(K2(), T(), N(), N()) : f(K2(), N(), N(), N());
  if (l.wing) return f(K2(), T(), T(), T());
  return l.grad ? f(K2(), T(), T(), N()) : f(K2(), N(), T(), N());
}

// Name of the kernel of the call's last launch (for the many-candidate gradient: the gradient launch, after
// the selection launch <2, 0, 1>).
inline void reproj_kernel_name(const ReprojLaunch& L, char* name, size_t len) {
  const KernelLaunch& l = L.launch[L.n_launches - 1];
  if (L.form == REPROJ_TILE)
    snprintf(name, len, "bbd::reproj_kernel<%d, %d>", l.grad ? 1 : 0, L.keep ? 1 : 0);
  else if (L.form == REPROJ_PIPE)
    snprintf(name, len, "bbd::reproj_pipe_kernel<%d, %d>", L.k, l.grad ? 1 : 0);
  else
    snprintf(name, len, "bbd::reproj_stream%s_kernel<%d, %d, %d%s>", L.tma ? "_tma" : "", L.k, l.grad ? 1 : 0, l.multi ? 1 : 0,
             l.wing ? ", 1" : "");
}

// ---- identity pre-pass ------------------------------------------------------------------------
struct IdentLaunch {
  bool stream;  // one warp per strip segment (ident_stream_kernel); otherwise the tile kernel over SCfg tiles
  int seg_rows, units;
};
inline IdentLaunch ident_launch(const bbd_ident_args& a, int sms) {
  IdentLaunch L = {false, 0, 0};
  if (a.force_tile) return L;
  L.stream = true;
  L.seg_rows = ident_seg_rows(a.height, a.width, a.batch, sms * 16);
  L.units = a.batch * IdentGeo::strips(a.width) * ((a.height + L.seg_rows - 1) / L.seg_rows);
  return L;
}

// ---- smoothness scratch ------------------------------------------------------------------------
// partial-sum slots (levels,B,4,parts) + the per-sample scalars (levels,B,2) + the ticket of the last-block reduction
struct SmoothLayout {
  int max_parts;  // partial-sum slots per (level, sample, quantity)
  size_t scalars, ticket, floats;  // offsets (floats) of the per-sample scalars and of the ticket; total size
};
inline SmoothLayout smooth_layout(int batch, int levels, const int32_t* h, const int32_t* w) {
  SmoothLayout L;
  L.max_parts = 1;
  for (int l = 0; l < levels; ++l) {
    const int c = sm_chunks(h[l], w[l]) > smr_blocks(h[l], w[l]) ? sm_chunks(h[l], w[l]) : smr_blocks(h[l], w[l]);
    L.max_parts = c > L.max_parts ? c : L.max_parts;
  }
  L.scalars = (size_t)levels * batch * 4 * L.max_parts;
  L.ticket = L.scalars + (size_t)levels * batch * 2;
  L.floats = L.ticket + 4;
  return L;
}

// ---- disparity backward -------------------------------------------------------------------------
// Every level in one launch (no scratch plane) when each has a supported factor and two full-resolution rows of
// tent sums fit the shared memory; otherwise the two-pass form.  The single launch reads gdepth and depth 16 bytes
// at a time and stores the gradient of a full-resolution (factor 1) level as float4s: those buffers must be 16-byte
// aligned.  (It reads gsmooth one element at a time.)
inline bool d2d_single_launch(const bbd_d2d_args& a) {
  bool fused = aligned16(a.gdepth) && aligned16(a.depth) && 2 * (size_t)a.width * sizeof(float) <= 48 * 1024;
  for (int l = 0; l < a.levels; ++l) {
    const int f = d2d_fused_factor(a, l);
    fused = fused && f != 0 && (f != 1 || aligned16(a.gdisp[l]));
  }
  return fused;
}

}  // namespace bbd
