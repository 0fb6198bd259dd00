/*
 * bbd_loss.h -- C ABI of libbbd_loss.so: the B200-native view-synthesis loss.
 *
 * The reference (kieran514/baseboostdepth) is pure PyTorch and ships no native
 * interface; what this library replaces is the chain of ATen calls issued by
 *   layers.py:160-167   BackprojectDepth.forward
 *   layers.py:181-195   Project3D.forward
 *   trainer.py:439,442  F.grid_sample(bilinear, border, align_corners=True)
 *   layers.py:235-249   SSIM.forward
 *   trainer.py:477-486  Trainer.compute_reprojection_loss
 *   trainer.py:508-557  identity terms, noise, per-pixel minimum (+ x_min_opt :983-1100)
 *   layers.py:203-216   get_smooth_loss (+ mean-normalisation trainer.py:560-562)
 *   trainer.py:456-460  F.interpolate(disp) + disp_to_depth (layers.py:13-22)
 * Each entry point below cites the reference lines it stands in for.
 *
 * Contract
 *   - All pointers are DEVICE pointers to fp32 (or the stated integer type),
 *     contiguous NCHW unless said otherwise; the caller allocates every
 *     input, output, gradient and scratch buffer.  The library never
 *     allocates or frees device memory and keeps no global state besides the
 *     last error string (thread-local).
 *   - All work is enqueued on `stream`; nothing synchronises; every call is
 *     CUDA-graph capturable.  One process drives one GPU.
 *   - Return value: 0 on success, a cudaError_t (>0) if a launch failed, or a
 *     negative BBD_E_* code for a bad argument.  Nothing throws, nothing exits.
 *   - There is no CPU implementation behind these symbols.
 *   - Alignment: every pointer must be aligned to its element type (4 bytes for float and int32).  Where a
 *     kernel can move 16 bytes at a time it checks the pointer first and falls back to narrower accesses when
 *     the address is not 16-byte aligned (the fused loss's TMA staging of target / depth / ident_min, the
 *     disparity -> depth forward's depth stores, the single-launch disparity backward's gdepth / depth loads and
 *     full-resolution gdisp stores, bbd_pack_rgba's planar loads, bbd_u8_to_f32).  The one exception is the
 *     channel-interleaved frame copies (frames_rgba, the rgba output of bbd_pack_rgba), which are only ever
 *     accessed one 16-byte pixel at a time: a non-NULL entry that is not 16-byte aligned is rejected with
 *     BBD_E_ARG.  Buffers from cudaMalloc or the PyTorch allocator always satisfy this.
 */
#ifndef BBD_LOSS_H_
#define BBD_LOSS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BBD_ABI_VERSION 2
#define BBD_MAX_FRAMES 16 /* image stacks: frames -7..7 and 's' */
#define BBD_MAX_GROUPS 8  /* noise stacks: one per baseline group */
#define BBD_MAX_REP 12    /* warped candidates per target sample (x_min_opt, decomp) */
#define BBD_MAX_IDENT 6   /* identity candidates per target sample */
#define BBD_MAX_SCALES 4

#define BBD_E_ARG (-1)   /* null pointer / negative size (or a size below the stated minimum) */
#define BBD_E_RANGE (-2) /* table entry or size outside the supported range */

typedef void* bbd_stream_t; /* cudaStream_t */

/* Per-batch index tables built on the host (baseboostdepth_b200/plan.py):
 *   hdr   (B,4)  int32: n_rep, n_ident, noise stack, noise row
 *   rep   (B,BBD_MAX_REP,4)   int32: frame stack, stack row, pose row, K row
 *   ident (B,BBD_MAX_IDENT,2) int32: frame stack, stack row
 * They replace the boolean-list masks of Trainer.valid_frames_trimin
 * (trainer.py:888-981) and the tensor copies of trainer.py:426-429,501-540. */
typedef struct bbd_tables {
  const int32_t* hdr;
  const int32_t* rep;
  const int32_t* ident;
} bbd_tables;

/* ---- identity pre-pass ---------------------------------------------------
 * trainer.py:501-523: identity_reprojection_losses[f] = compute_reprojection_loss(
 * color[f], color[0]) for every source of a sample, + noise, then the minimum
 * over them in candidate order.  Writes ident_min (B,H,W) = min_j(ident_j +
 * noise*noise_scale) and ident_arg (B,H,W) uint8 = first j attaining it. */
typedef struct bbd_ident_args {
  int32_t batch, height, width;
  int32_t no_ssim; /* options.py:173 */
  const float* target;                   /* ("color",0,0): (B,3,H,W) */
  const float* frames[BBD_MAX_FRAMES];   /* ("color",f,0) stacks: (n_f,3,H,W) */
  const float* noise[BBD_MAX_GROUPS];    /* randn planes per group: (n_g,1,H,W) */
  float noise_scale;                     /* 1e-5 for raw randn, 1 if pre-scaled */
  bbd_tables tab;
  float* ident_min;
  uint8_t* ident_arg;
  /* Optional: (n_f,H,W,4) channel-interleaved copies of the frame stacks, written as a by-product (every
   * source row passes through registers here anyway); the layout bbd_reproj_args.frames_rgba expects.
   * NULL entries are skipped; a non-NULL entry must be 16-byte aligned (BBD_E_ARG otherwise). */
  float* frames_rgba[BBD_MAX_FRAMES];
  int32_t force_tile; /* 0: streaming form (contracted / separable arithmetic); != 0: tile kernel with the
                         reference's rounding, no copies written */
} bbd_ident_args;
int bbd_ident_forward(const bbd_ident_args* a, bbd_stream_t stream);

/* ---- fused reprojection loss, forward + backward in one pass -------------
 * trainer.py:444-475 (generate_images_pred) and :525-557 (compute_losses) for
 * all scales of a step: back-project, project with P = (K@T)[:3], bilinear
 * border warp of every candidate source, SSIM + L1 mix, per-pixel minimum
 * against ident_min, and -- because the loss is a mean with a known weight --
 * the gradient of sum_s mean(to_optimise_s) with respect to depth and P.
 * Outputs are per-tile partial sums; bbd_reproj_finalize reduces them in a
 * fixed order (deterministic, no float atomics). */
typedef struct bbd_reproj_args {
  int32_t batch, height, width, num_scales;
  int32_t no_ssim;
  int32_t need_grad;  /* 0: forward only (validation / logging) */
  int32_t max_rep;    /* max n_rep over the batch (sizes shared memory) */
  int32_t num_pose;   /* rows of P */
  const float* target;                 /* (B,3,H,W) */
  const float* frames[BBD_MAX_FRAMES]; /* stacks (n_f,3,H,W) */
  const float* depth;                  /* (S,B,H,W) outputs[("depth",0,s)] */
  const float* inv_K;                  /* (B,4,4) inputs[("inv_K",0)] */
  const float* P;                      /* (num_pose,3,4) = (K@T)[:, :3, :] */
  const float* ident_min;              /* (B,H,W) from bbd_ident_forward */
  bbd_tables tab;
  float* loss_part;   /* (S,B,tiles) partial sums of to_optimise */
  float* gpose_part;  /* (S,B,BBD_MAX_REP,tiles,12) partial d/dP sums; may be NULL if !need_grad */
  float* gdepth;      /* (S,B,H,W) d mean_s / d depth_s;        may be NULL if !need_grad */
  uint8_t* winner;    /* (S,B,H,W) argmin index in candidate order (reproj..., then ident...); may be NULL.  With
                       * max_rep > 2 and need_grad a non-NULL plane lets the call run as a forward-only selection
                       * launch followed by a gradient launch that reads the winners from here (faster) */
  const uint8_t* ident_arg; /* (B,H,W); only read when winner != NULL */
  /* Optional channel-interleaved copies of the frame stacks, (n_f,H,W,4) = r,g,b,0 per pixel, written by
   * bbd_pack_rgba: one 16-byte load fetches a bilinear tap of all three channels.  When every stack
   * that the tables reference has one, and 1 <= min_rep <= max_rep <= 2, bbd_reproj_fused runs the
   * streaming kernel (csrc/bbd_stream.cuh); otherwise the tile kernel, which reads `frames`.  Every non-NULL
   * entry must be 16-byte aligned (BBD_E_ARG otherwise). */
  const float* frames_rgba[BBD_MAX_FRAMES];
  int32_t min_rep;    /* min n_rep over the batch (0 = unknown: tile kernel) */
  /* Optional fused finalize (streaming kernel only; see bbd_reproj_finalizes_itself): when `tickets` is set the
   * last warp of every (scale, sample) reduces that pair's partials in a fixed order and the results land in
   * loss_out (S) / gpose_out (S,num_pose,3,4) without a second launch.  tickets: S*B + S int32, zero before the
   * first launch (the kernel leaves them zero); pair_sum: S*B floats of scratch.  gpose_out rows that no
   * candidate references are not written (zero them once). */
  int32_t* tickets;
  float* pair_sum;
  float* loss_out;
  float* gpose_out;
  int32_t force_tile; /* != 0: always the tile kernel (exact-rounding arithmetic), for A/B measurements */
} bbd_reproj_args;
int bbd_reproj_tiles(int32_t height, int32_t width); /* partial-sum slots per (scale, sample) */
/* The projection chain of the streaming kernel on its own (parity instrumentation): for sample i < n, with
 * inv_K row i and P row i, grid (n,2,H,W) = what Project3D.forward returns (layers.py:181-195, permuted),
 * pix (n,2,H,W) = the clipped source coordinates of F.grid_sample (align_corners=True, border); floor(pix)
 * is the north-west bilinear tap.  Either output may be NULL. */
int bbd_project_coords(int32_t n, int32_t height, int32_t width, const float* depth, const float* inv_K, const float* P,
                       float* grid, float* pix, bbd_stream_t stream);
/* (n,3,H,W) planar -> (n,H,W,4) interleaved, 4th component 0: the gather layout of the streaming kernel.
 * rgba must be 16-byte aligned (BBD_E_ARG otherwise); planar may start anywhere. */
int bbd_pack_rgba(int32_t n, int32_t height, int32_t width, const float* planar, float* rgba, bbd_stream_t stream);
int bbd_reproj_fused(const bbd_reproj_args* a, bbd_stream_t stream);
/* 1 if bbd_reproj_fused, for these arguments, also performs the reduction of bbd_reproj_finalize (tickets given
 * and the streaming kernel is selected); the caller then skips bbd_reproj_finalize. */
int bbd_reproj_finalizes_itself(const bbd_reproj_args* a);
/* Symbol (as ncu / nsys print it) of the kernel bbd_reproj_fused launches for these arguments. */
const char* bbd_reproj_kernel_name(const bbd_reproj_args* a);
/* loss (S) = sum(loss_part)/(B*H*W); gpose (S,num_pose,3,4) = sum over tiles. */
int bbd_reproj_finalize(const bbd_reproj_args* a, float* loss, float* gpose, bbd_stream_t stream);

/* ---- gradient of the fused loss w.r.t. the colour frames -------------------
 * trainer.py:477-486 + :525-557 under autograd with the target ("color",0,0) and the source stacks
 * ("color",f,0) requiring grad: only the per-pixel winner's photometric term is differentiated, the winners
 * being the ones the forward wrote to bbd_reproj_args.winner (which, with ident_arg, this needs; depth, inv_K,
 * P, target, frames and tab as in the forward).  Two calls around a caller-side STABLE sort:
 *   bbd_frame_grad         writes gtarget, gident, gpred and keys (coef is scratch);
 *   (caller)               sorts keys -> keys_sorted with order = the permutation as int32 (n_items entries);
 *   bbd_frame_grad_stacks  gathers, per stack pixel, the transposed bilinear warps of every scale, candidate
 *                          and decomp twin that sampled it (four runs of the sorted order, as
 *                          bbd_grid_sample_backward_image) plus the identity-source gradients; seg_start is
 *                          scratch.  Every gframes[f] given is fully written (zero where nothing reads it).
 * Sums run in a fixed order and use no atomics: the result is bit-reproducible.
 * n_items = num_scales*B*max_rep*H*W; n_keys = (sum of stack_rows)*H*W; both must stay below 2^31. */
typedef struct bbd_frame_grad_args {
  const float* gscale;                  /* (S) device: upstream gradient of the per-scale reprojection means */
  int32_t stack_rows[BBD_MAX_FRAMES];   /* rows of each frame stack (0 for an empty or absent slot) */
  float* coef;                          /* (S,B,3,6,H,W) scratch; may be NULL under no_ssim */
  float* gpred;                         /* (S,B,max_rep,3,H,W): d loss / d warped candidate (read where keyed) */
  int32_t* keys;                        /* (n_items): stack row * H*W + north-west tap, or n_keys (no gradient) */
  float* gident;                        /* (B,BBD_MAX_IDENT,3,H,W): identity-source gradients, rows < n_ident */
  float* gtarget;                       /* (B,3,H,W) or NULL */
  const int32_t* keys_sorted;           /* bbd_frame_grad_stacks only: (n_items) */
  const int32_t* order;                 /* bbd_frame_grad_stacks only: (n_items) */
  int32_t* seg_start;                   /* bbd_frame_grad_stacks only: n_keys + 1 int32 of scratch */
  float* gframes[BBD_MAX_FRAMES];       /* bbd_frame_grad_stacks only: (stack_rows[f],3,H,W) or NULL to skip */
} bbd_frame_grad_args;
int bbd_frame_grad(const bbd_reproj_args* a, const bbd_frame_grad_args* f, bbd_stream_t stream);
int bbd_frame_grad_stacks(const bbd_reproj_args* a, const bbd_frame_grad_args* f, bbd_stream_t stream);

/* ---- camera motion from network outputs ---------------------------------------
 * layers.py:25-100: transformation_from_parameters(axisangle, translation, invert) =
 * get_translation_matrix(t) @ rot_from_axisangle(v), or R^T @ T(-t) when invert.  One thread per
 * pose instead of ~40 tiny tensor kernels; the backward propagates forward-mode tangents through
 * the same formulas.  axisangle, translation: (n,3); T: (n,4,4). */
int bbd_pose_forward(int32_t n, const float* axisangle, const float* translation, int32_t invert, float* T,
                     bbd_stream_t stream);
int bbd_pose_backward(int32_t n, const float* axisangle, const float* translation, int32_t invert,
                      const float* gT, float* gaxisangle, float* gtranslation, bbd_stream_t stream);

/* ---- projection matrices -----------------------------------------------------
 * layers.py:182: P = (K @ T)[:, :3, :] for every pose row, K row given per pose (the trainer
 * pairs a frame's poses with K[:n], trainer.py:431).  Each element follows the rounding of
 * ATen's CPU bmm for tiny matrices (multiply, add, k ascending; bit-identical to it).  backward: gT = K[:3,:]^T @ gP (rows 0..3). */
int bbd_pose_pack_forward(int32_t n_pose, const float* K /* (B,4,4) */, const int32_t* k_row /* (n_pose) */,
                          const float* T /* (n_pose,4,4) */, float* P /* (n_pose,3,4) */, bbd_stream_t stream);
int bbd_pose_pack_backward(int32_t n_pose, const float* K, const int32_t* k_row, const float* gP /* (n_pose,3,4) */,
                           float* gT /* (n_pose,4,4) */, bbd_stream_t stream);

/* ---- warped images on demand ----------------------------------------------
 * outputs[("color",f,s)] for logging (trainer.py:722-726): same projection and
 * sampling as bbd_reproj_fused for one frame stack; pose rows / K rows are the
 * first n rows (the trainer's [:frame_size] slices, trainer.py:431-432). */
int bbd_warp_forward(int32_t n, int32_t height, int32_t width, const float* images, /* (n,3,H,W) */
                     const float* depth,                                           /* (n,1,H,W) */
                     const float* inv_K, const float* P, float* warped,             /* (n,3,H,W) */
                     float* grid /* (n,2,H,W) normalised coords, may be NULL */, bbd_stream_t stream);

/* ---- edge-aware smoothness, forward + backward ----------------------------
 * trainer.py:560-563 + layers.py:203-216 for every pyramid level of a step:
 * d = disp / (mean_hw(disp) + 1e-7); loss = mean|dx d|e^{-mean_c|dx I|} + same in y.
 * Two enqueued stages (sample means; per-pixel terms, coupling sums and the level losses), each covering
 * all levels, plus a small element-wise finish unless the caller defers it (defer_norm).  loss[l] and gdisp[l] = d loss[l] / d disp_l
 * are unweighted; the caller applies disparity_smoothness / 2^scale (trainer.py:564). */
typedef struct bbd_smooth_args {
  int32_t batch, levels;
  int32_t h[BBD_MAX_SCALES], w[BBD_MAX_SCALES];
  const float* disp[BBD_MAX_SCALES]; /* (B,1,h,w) outputs[("disp",s)] */
  const float* img[BBD_MAX_SCALES];  /* (B,3,h,w) inputs[("color",0,s)] */
  float* gdisp[BBD_MAX_SCALES];      /* (B,1,h,w) or NULL for forward only */
  float* scratch;                    /* bbd_smooth_scratch_floats() floats */
  float* loss;                       /* (levels) */
  int32_t max_chunks;                /* set by the library */
  int32_t normalize;                 /* 1: divide by the per-sample mean first (trainer.py:560-562);
                                        0: plain get_smooth_loss(disp, img) (layers.py:203-216) */
  int32_t defer_norm;                /* 1: leave gdisp[l] = d loss / d(normalised disp) and write the two scalars per
                                        (level, sample) that finish it, g_disp = g * coef[0] - coef[1], to `coef`;
                                        bbd_disp_to_depth_backward applies them on the fly (gsmooth_coef) */
  float* coef;                       /* (levels,B,2); required when defer_norm */
} bbd_smooth_args;
size_t bbd_smooth_scratch_floats(int32_t batch, int32_t levels, const int32_t* h, const int32_t* w);
int bbd_smooth_fused(const bbd_smooth_args* a, bbd_stream_t stream);
/* Gradient of the smoothness terms w.r.t. the colour levels (layers.py:203-216 under autograd): per pixel, a
 * gather over its four edges.  gimg[l] = gscale[l] * d loss[l] / d img_l, with the normalisation scalar
 * 1/(mean+1e-7) read from coef[l,b,0] as bbd_smooth_fused leaves it (defer_norm), or 1 when coef is NULL. */
typedef struct bbd_smooth_img_args {
  int32_t batch, levels;
  int32_t h[BBD_MAX_SCALES], w[BBD_MAX_SCALES];
  const float* disp[BBD_MAX_SCALES]; /* (B,1,h,w) */
  const float* img[BBD_MAX_SCALES];  /* (B,3,h,w) */
  const float* coef;                 /* (levels,B,2) or NULL */
  const float* gscale;               /* (levels) device: upstream gradient of each level's loss */
  float* gimg[BBD_MAX_SCALES];       /* (B,3,h,w), or NULL to skip the level */
} bbd_smooth_img_args;
int bbd_smooth_image_grad(const bbd_smooth_img_args* a, bbd_stream_t stream);

/* ---- disparity -> full-resolution depth, and back ---------------------------
 * trainer.py:456-461 for every scale of a step: F.interpolate(bilinear,
 * align_corners=False) to (H,W), then depth = 1/(min_disp + (max_disp-min_disp)*disp)
 * (layers.py:13-22); sql != 0 skips the conversion (opt.SQL).  The backward gathers,
 * for every low-resolution disparity pixel, the full-resolution pixels it contributed
 * to (no atomics) and multiplies by gscale[s] (a DEVICE array: the upstream gradient of
 * the per-scale loss is only known on the device when autograd runs). */
typedef struct bbd_d2d_args {
  int32_t batch, levels, height, width;
  int32_t h[BBD_MAX_SCALES], w[BBD_MAX_SCALES];
  float min_disp;  /* float(1/max_depth)               (layers.py:18) */
  float disp_span; /* float(1/min_depth - 1/max_depth) (layers.py:20, formed in double like the reference) */
  int32_t sql;
  const float* disp[BBD_MAX_SCALES]; /* (B,1,h,w) */
  float* depth;                      /* (S,B,H,W) written by forward, read by backward */
  const float* gdepth;               /* (S,B,H,W) backward only */
  const float* gscale;               /* (S) device, backward only */
  const float* gsmooth[BBD_MAX_SCALES]; /* (B,1,h,w) optional extra term (smoothness gradient), or NULL */
  const float* gsmooth_scale;        /* (S) device: gdisp += gsmooth_scale[s] * gsmooth[s] */
  const float* gsmooth_coef;         /* (S,B,2) or NULL: gsmooth[s] is first finished as g * coef[0] - coef[1]
                                        (bbd_smooth_args.defer_norm) */
  float* gdisp[BBD_MAX_SCALES];      /* (B,1,h,w) backward only */
  float* scratch;                    /* backward only: bbd_d2d_scratch_floats() floats (row sums of the
                                        separable gather for the levels upsampled by 2, 4 or 8) */
} bbd_d2d_args;
size_t bbd_d2d_scratch_floats(const bbd_d2d_args* a);
int bbd_disp_to_depth_forward(const bbd_d2d_args* a, bbd_stream_t stream);
int bbd_disp_to_depth_backward(const bbd_d2d_args* a, bbd_stream_t stream);
/* The two passes of bbd_disp_to_depth_backward on their own, for callers that overlap them on streams:
 * pass 1 reduces gdepth along rows into `scratch` for the levels with an integer factor 2/4/8 (it needs
 * neither the upstream scalars nor the smoothness gradient); pass 2 finishes the levels
 * [level_begin, level_end) -- a level at full resolution does not read `scratch`, so its pass 2 can run
 * next to pass 1. */
int bbd_disp_to_depth_backward_pass1(const bbd_d2d_args* a, bbd_stream_t stream);
int bbd_disp_to_depth_backward_pass2(const bbd_d2d_args* a, int32_t level_begin, int32_t level_end,
                                     bbd_stream_t stream);

/* ---- module-level operators (tier A: trainer.py unchanged) -----------------
 * Same maths as the layers in layers.py, one kernel each, forward and backward.
 * Sizes (here and for bbd_project_coords, bbd_pack_rgba, bbd_pose_* and bbd_pose_pack_*): n == 0 is a
 * no-op that returns 0 and touches nothing (an empty sub-batch of the trainer reaches these calls); a negative
 * count, channel count or size is BBD_E_ARG; H*W, Ho*Wo or n*channels above INT32_MAX is BBD_E_RANGE. */
/* layers.py:160-167; points (n,4,HW) */
int bbd_backproject_forward(int32_t n, int32_t height, int32_t width, const float* depth,
                            const float* inv_K, float* points, bbd_stream_t stream);
int bbd_backproject_backward(int32_t n, int32_t height, int32_t width, const float* inv_K,
                             const float* gpoints, float* gdepth, bbd_stream_t stream);
/* layers.py:181-195 after P=(K@T)[:3]; pix laid out (n,2,H,W) -- the reference returns the
 * (n,H,W,2) permuted view of exactly this memory. */
int bbd_project_forward(int32_t n, int32_t height, int32_t width, const float* points, const float* P,
                        float eps, float* pix, bbd_stream_t stream);
/* gpoints (n,4,HW); gP_part (n,chunks,12) reduced by the caller; chunks = bbd_project_chunks */
int bbd_project_chunks(int32_t height, int32_t width);
int bbd_project_backward(int32_t n, int32_t height, int32_t width, const float* points, const float* P,
                         float eps, const float* gpix, float* gpoints, float* gP_part,
                         bbd_stream_t stream);
/* trainer.py:442 / :439: F.grid_sample(images, grid, align_corners=True, padding_mode="border"),
 * bilinear.  images (n,C,H,W); grid laid out (n,2,Ho,Wo) -- the permuted memory Project3D returns;
 * out (n,C,Ho,Wo).  backward: gradient w.r.t. the grid (per-pixel gather, deterministic); the gradient
 * w.r.t. the sampled images -- never requested by the trainer -- is the pair of calls further down. */
int bbd_grid_sample_forward(int32_t n, int32_t channels, int32_t height, int32_t width, int32_t out_h,
                            int32_t out_w, const float* images, const float* grid, float* out,
                            bbd_stream_t stream);
int bbd_grid_sample_backward(int32_t n, int32_t channels, int32_t height, int32_t width, int32_t out_h,
                             int32_t out_w, const float* images, const float* grid, const float* gout,
                             float* ggrid /* (n,2,Ho,Wo) */, bbd_stream_t stream);
/* Gradient of F.grid_sample w.r.t. `images` (trainer.py:442 under autograd; ATen grid_sampler_2d_backward scatters it
 * with atomic adds).  Atomics-free and bit-reproducible: bbd_grid_sample_dest_keys writes, for every output
 * (n, o) in order, the key n*H*W + (linear index of its north-west tap); the caller sorts the keys with a STABLE
 * sort (keys_sorted, order = the permutation, as int32); bbd_grid_sample_backward_image then gathers, per source
 * pixel, the outputs that touch it from four contiguous runs of that order.  seg_start: n*H*W + 1 int32 of
 * scratch.  gimages (n,C,H,W) is fully written. */
int bbd_grid_sample_dest_keys(int32_t n, int32_t height, int32_t width, int32_t out_h, int32_t out_w,
                              const float* grid, int32_t* keys, bbd_stream_t stream);
int bbd_grid_sample_backward_image(int32_t n, int32_t channels, int32_t height, int32_t width, int32_t out_h,
                                   int32_t out_w, const float* grid, const float* gout,
                                   const int32_t* keys_sorted, const int32_t* order, int32_t* seg_start,
                                   float* gimages, bbd_stream_t stream);
/* layers.py:235-249; gx / gy may be NULL; height and width >= 2 (reflection padding), BBD_E_RANGE otherwise */
int bbd_ssim_forward(int32_t n, int32_t channels, int32_t height, int32_t width, const float* x,
                     const float* y, float* out, bbd_stream_t stream);
int bbd_ssim_backward(int32_t n, int32_t channels, int32_t height, int32_t width, const float* x,
                      const float* y, const float* gout, float* gx, float* gy, bbd_stream_t stream);

/* Loss assembly, trainer.py:557-570: per_scale[s] = reproj[s] + weight[s] * smooth[s]
 * (weight[s] = disparity_smoothness / 2^s), total = (((p0 + p1) + p2) + ...) / num_scales -- one launch
 * instead of a handful of 4-element tensor kernels.  backward: g_total (1 float, may be NULL),
 * g_per_scale (S floats, may be NULL) -> g_reproj[S], g_smooth[S] (the upstream scalars the fused
 * loss's backward consumes).  All pointers are device memory. */
int bbd_loss_combine_forward(int32_t num_terms, const float* reproj, const float* smooth, const float* weight,
                             float num_scales, float* per_scale, float* total, bbd_stream_t stream);
int bbd_loss_combine_backward(int32_t num_terms, const float* g_total, const float* g_per_scale, const float* weight,
                              float num_scales, float* g_reproj, float* g_smooth, bbd_stream_t stream);

/* Frames as decoded (8-bit) -> the fp32 tensors the reference's loader hands the trainer:
 * torchvision ToTensor = uint8 -> float32, IEEE division by 255 (datasets/mono_dataset.py:55,201-203).
 * dst[i] = (float)src[i] / 255 for i < n, bit-identical to ToTensor.  Lets a batch cross PCIe at
 * one byte per colour sample instead of four (staging.BatchStager). */
int bbd_u8_to_f32(const uint8_t* src, float* dst, size_t n, bbd_stream_t stream);

int bbd_version(void);
const char* bbd_last_error_string(void);

#ifdef __cplusplus
}
#endif
#endif /* BBD_LOSS_H_ */
