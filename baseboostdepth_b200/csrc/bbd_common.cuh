// Shared host/device building blocks of the view-synthesis loss kernels.
//
// Everything here is `__host__ __device__` so that the very same code the
// sm_100a kernels run can be stepped on the CPU by tests/emu (a test-only
// harness that executes one thread block phase by phase).  The product is the
// CUDA build; the host instantiation exists only under tests/.
//
// Rounding discipline: the reference evaluates this path as a chain of separate
// fp32 ATen kernels, i.e. every elementary operation is rounded on its own and
// nothing is contracted across tensor ops, except inside bmm (a k-sequential
// FMA chain, checked bit-for-bit against torch CPU) and inside grid_sample's
// 4-tap accumulation.  The helpers below therefore use the explicitly rounded
// intrinsics (never contracted by nvcc) and FMA only where the reference has it.
#pragma once
#include <assert.h>
#include <math.h>
#include <stdint.h>

#include "../../include/bbd_loss.h"

#if defined(__CUDACC__)
#define BBD_HD __host__ __device__ __forceinline__
#else
#define BBD_HD inline
#endif

namespace bbd {

#if defined(__CUDA_ARCH__)
BBD_HD float mul(float a, float b) { return __fmul_rn(a, b); }
BBD_HD float add(float a, float b) { return __fadd_rn(a, b); }
BBD_HD float sub(float a, float b) { return __fsub_rn(a, b); }
BBD_HD float fma_(float a, float b, float c) { return __fmaf_rn(a, b, c); }
BBD_HD float div_(float a, float b) { return __fdiv_rn(a, b); }
BBD_HD float rcp_rn(float a) { return __frcp_rn(a); }  // correctly rounded 1/a (== 1.0f / a, fewer instructions)
BBD_HD float rcp_approx(float a) { return __fdividef(1.0f, a); }  // gradients only (<= 2 ulp)
#else
// host build is compiled with -ffp-contract=off
BBD_HD float mul(float a, float b) { return a * b; }
BBD_HD float add(float a, float b) { return a + b; }
BBD_HD float sub(float a, float b) { return a - b; }
BBD_HD float fma_(float a, float b, float c) { return fmaf(a, b, c); }
BBD_HD float div_(float a, float b) { return a / b; }
BBD_HD float rcp_rn(float a) { return 1.0f / a; }
BBD_HD float rcp_approx(float a) { return 1.0f / a; }
#endif

// a / d for a fixed divisor d with y = RN(1/d): q = RN(a*y); r = a - d*q (exact, FMA);
// RN(q + r*y) is the correctly rounded quotient (Markstein).  Three instructions instead of
// the IEEE division subroutine; equality with a / d is checked exhaustively over all 2^23
// significands for the divisors used here (9, W-1, H-1) in tests/test_division.py.
BBD_HD float div_const(float a, float d, float y) {
  const float q = mul(a, y);
  const float r = fma_(-d, q, a);
  return fma_(r, y, q);
}

// ---- two values per lane -------------------------------------------------------------------
// sm_100 issues packed fp32x2 multiply / add / fma (FMUL2, FADD2, FFMA2) with the same rounding as
// the scalar forms at half the issue slots per value (scripts/micro/ffma2_bench.cu: packed
// mul+add runs at 2x the scalar rate).  The statistics phase processes two rows per thread this way.
struct f2 {
  float x, y;
};
BBD_HD f2 mk2(float x, float y) { f2 r; r.x = x; r.y = y; return r; }
BBD_HD f2 bc2(float v) { return mk2(v, v); }
#if defined(__CUDA_ARCH__)
BBD_HD float2 as_f2(const f2& a) { return make_float2(a.x, a.y); }
BBD_HD f2 from_f2(const float2& a) { return mk2(a.x, a.y); }
BBD_HD f2 mul(const f2& a, const f2& b) { return from_f2(__fmul2_rn(as_f2(a), as_f2(b))); }
BBD_HD f2 add(const f2& a, const f2& b) { return from_f2(__fadd2_rn(as_f2(a), as_f2(b))); }
BBD_HD f2 fma_(const f2& a, const f2& b, const f2& c) { return from_f2(__ffma2_rn(as_f2(a), as_f2(b), as_f2(c))); }
BBD_HD f2 sub(const f2& a, const f2& b) { return from_f2(__fadd2_rn(as_f2(a), make_float2(-b.x, -b.y))); }
#else
BBD_HD f2 mul(const f2& a, const f2& b) { return mk2(a.x * b.x, a.y * b.y); }
BBD_HD f2 add(const f2& a, const f2& b) { return mk2(a.x + b.x, a.y + b.y); }
BBD_HD f2 fma_(const f2& a, const f2& b, const f2& c) { return mk2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
BBD_HD f2 sub(const f2& a, const f2& b) { return mk2(a.x - b.x, a.y - b.y); }
#endif
BBD_HD f2 div_(const f2& a, const f2& b) { return mk2(div_(a.x, b.x), div_(a.y, b.y)); }
BBD_HD f2 div_const(const f2& a, float d, float y) {
  const f2 q = mul(a, bc2(y));
  const f2 r = fma_(bc2(-d), q, a);
  return fma_(r, bc2(y), q);
}

// 16 bytes through the read-only path
struct f4 {
  float x, y, z, w;
};
BBD_HD f4 load4(const float* p) {
#if defined(__CUDA_ARCH__)
  const float4 v = __ldg(reinterpret_cast<const float4*>(p));
  f4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w;
  return r;
#else
  assert(((uintptr_t)p & 15) == 0 && "load4: a 16-byte load needs a 16-byte aligned address");
  f4 r; r.x = p[0]; r.y = p[1]; r.z = p[2]; r.w = p[3];
  return r;
#endif
}

// SSIM constants (layers.py:232-233), photometric mix (trainer.py:485)
#define BBD_C1 0.0001f
#define BBD_C2 0.0009f
#define BBD_W_SSIM 0.85f
#define BBD_W_L1 0.15f
#define BBD_THIRD 0.3333333432674407958984375f /* float(1/3): ATen CUDA mean = sum * factor */

// Reflection padding by one pixel (layers.py:230): -1 -> 1, n -> n-2.  Coordinates two
// outside the image are never consumed by a valid window; they are folded the same way
// and finally clamped so that every address stays inside the plane.
BBD_HD int reflect1(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  if (i < 0) i = 0;
  if (i >= n) i = n - 1;
  return i;
}

// Rows [:3,:3] of a row-major 4x4 inverse intrinsics and a row-major 3x4 projection.
struct Cam {
  float ik[9];
  float p[12];
  float wm1, hm1, rw, rh;  // W-1, H-1 and their correctly rounded reciprocals
};

BBD_HD void load_cam(Cam& c, const float* inv_K4x4, const float* P3x4, int W, int H) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) c.ik[i * 3 + j] = inv_K4x4[i * 4 + j];
  for (int i = 0; i < 12; ++i) c.p[i] = P3x4[i];
  c.wm1 = (float)(W - 1);
  c.hm1 = (float)(H - 1);
  c.rw = div_(1.0f, c.wm1);
  c.rh = div_(1.0f, c.hm1);
}

// Everything the bilinear tap needs, and (for the backward) the partials of it.
struct Sample {
  float ix, iy;      // clipped source coordinates
  float mx, my;      // clip gradient masks (0 on or outside the border)
  int x0, y0;        // north-west tap
  float X, Y, Z;     // camera-space point (depth * ray)
  float rx, ry, rz;  // ray = inv_K[:3,:3] @ (x, y, 1)
  float ux, uy, zz;  // projected pixel (before normalisation) and z + eps
};

// BackprojectDepth (layers.py:160-167) + Project3D (layers.py:181-195) + the coordinate
// part of grid_sample (ATen GridSampler: unnormalise, clip to the border) for one pixel.
BBD_HD void project_pixel(const Cam& c, int px, int py, float depth, int W, int H, Sample& s) {
  const float x = (float)px, y = (float)py;
  // bmm: acc = a0*b0; acc = fma(a1, b1, acc); acc = fma(a2, b2, acc)
  s.rx = fma_(c.ik[2], 1.0f, fma_(c.ik[1], y, mul(c.ik[0], x)));
  s.ry = fma_(c.ik[5], 1.0f, fma_(c.ik[4], y, mul(c.ik[3], x)));
  s.rz = fma_(c.ik[8], 1.0f, fma_(c.ik[7], y, mul(c.ik[6], x)));
  s.X = mul(depth, s.rx);
  s.Y = mul(depth, s.ry);
  s.Z = mul(depth, s.rz);
  const float cx = fma_(c.p[3], 1.0f, fma_(c.p[2], s.Z, fma_(c.p[1], s.Y, mul(c.p[0], s.X))));
  const float cy = fma_(c.p[7], 1.0f, fma_(c.p[6], s.Z, fma_(c.p[5], s.Y, mul(c.p[4], s.X))));
  const float cz = fma_(c.p[11], 1.0f, fma_(c.p[10], s.Z, fma_(c.p[9], s.Y, mul(c.p[8], s.X))));
  s.zz = add(cz, 1e-7f);
  s.ux = div_(cx, s.zz);
  s.uy = div_(cy, s.zz);
  // pix /= (W-1); (pix - 0.5) * 2   (layers.py:191-193)
  const float gx = mul(sub(div_const(s.ux, c.wm1, c.rw), 0.5f), 2.0f);
  const float gy = mul(sub(div_const(s.uy, c.hm1, c.rh), 0.5f), 2.0f);
  // grid_sampler_unnormalize(align_corners): ((g + 1) / 2) * (size - 1)
  float ix = mul(mul(add(gx, 1.0f), 0.5f), c.wm1);
  float iy = mul(mul(add(gy, 1.0f), 0.5f), c.hm1);
  // clip_coordinates_set_grad: the border itself counts as outside for the gradient
  const float wmax = c.wm1, hmax = c.hm1;
  if (!(ix > 0.0f)) { ix = 0.0f; s.mx = 0.0f; } else if (ix >= wmax) { ix = wmax; s.mx = 0.0f; } else { s.mx = 1.0f; }
  if (!(iy > 0.0f)) { iy = 0.0f; s.my = 0.0f; } else if (iy >= hmax) { iy = hmax; s.my = 0.0f; } else { s.my = 1.0f; }
  s.ix = ix;
  s.iy = iy;
  s.x0 = (int)floorf(ix);
  s.y0 = (int)floorf(iy);
}

// project_pixel for two pixels of one column (rows py0, py1) at once: the rounded multiply / add / fma
// chain runs on packed fp32x2 values (identical rounding per value), the two perspective divisions,
// the clip and the floor stay scalar.
BBD_HD void project_finish(const Cam& c, float ix, float iy, Sample& s) {
  const float wmax = c.wm1, hmax = c.hm1;
  if (!(ix > 0.0f)) { ix = 0.0f; s.mx = 0.0f; } else if (ix >= wmax) { ix = wmax; s.mx = 0.0f; } else { s.mx = 1.0f; }
  if (!(iy > 0.0f)) { iy = 0.0f; s.my = 0.0f; } else if (iy >= hmax) { iy = hmax; s.my = 0.0f; } else { s.my = 1.0f; }
  s.ix = ix;
  s.iy = iy;
  s.x0 = (int)floorf(ix);
  s.y0 = (int)floorf(iy);
}
BBD_HD void project_pixel2(const Cam& c, int px, int py0, int py1, float depth0, float depth1, Sample& s0, Sample& s1) {
  const float x = (float)px;
  const f2 y = mk2((float)py0, (float)py1), one = bc2(1.0f), d = mk2(depth0, depth1);
  const f2 rx = fma_(bc2(c.ik[2]), one, fma_(bc2(c.ik[1]), y, bc2(mul(c.ik[0], x))));
  const f2 ry = fma_(bc2(c.ik[5]), one, fma_(bc2(c.ik[4]), y, bc2(mul(c.ik[3], x))));
  const f2 rz = fma_(bc2(c.ik[8]), one, fma_(bc2(c.ik[7]), y, bc2(mul(c.ik[6], x))));
  const f2 X = mul(d, rx), Y = mul(d, ry), Z = mul(d, rz);
  const f2 cx = fma_(bc2(c.p[3]), one, fma_(bc2(c.p[2]), Z, fma_(bc2(c.p[1]), Y, mul(bc2(c.p[0]), X))));
  const f2 cy = fma_(bc2(c.p[7]), one, fma_(bc2(c.p[6]), Z, fma_(bc2(c.p[5]), Y, mul(bc2(c.p[4]), X))));
  const f2 cz = fma_(bc2(c.p[11]), one, fma_(bc2(c.p[10]), Z, fma_(bc2(c.p[9]), Y, mul(bc2(c.p[8]), X))));
  const f2 zz = add(cz, bc2(1e-7f));
  const f2 ux = div_(cx, zz), uy = div_(cy, zz);
  const f2 gx = mul(sub(div_const(ux, c.wm1, c.rw), bc2(0.5f)), bc2(2.0f));
  const f2 gy = mul(sub(div_const(uy, c.hm1, c.rh), bc2(0.5f)), bc2(2.0f));
  const f2 ix = mul(mul(add(gx, one), bc2(0.5f)), bc2(c.wm1));
  const f2 iy = mul(mul(add(gy, one), bc2(0.5f)), bc2(c.hm1));
  s0.rx = rx.x; s0.ry = ry.x; s0.rz = rz.x; s0.X = X.x; s0.Y = Y.x; s0.Z = Z.x; s0.zz = zz.x; s0.ux = ux.x; s0.uy = uy.x;
  s1.rx = rx.y; s1.ry = ry.y; s1.rz = rz.y; s1.X = X.y; s1.Y = Y.y; s1.Z = Z.y; s1.zz = zz.y; s1.ux = ux.y; s1.uy = uy.y;
  project_finish(c, ix.x, iy.x, s0);
  project_finish(c, ix.y, iy.y, s1);
}

// Bilinear taps of one channel plane (ATen grid_sampler_2d, bilinear): weights from the
// opposite corners, out-of-range taps contribute nothing, accumulation is an FMA chain.
struct Taps {
  float wnw, wne, wsw, wse;
  int onw, one, osw, ose;  // offsets into a channel plane
  bool bne, bsw, bse;      // tap inside the image (north-west always is after clipping)
};

BBD_HD void make_taps(const Sample& s, int W, int H, Taps& t) {
  const float fx0 = (float)s.x0, fy0 = (float)s.y0;
  const float fx1 = fx0 + 1.0f, fy1 = fy0 + 1.0f;
  t.wnw = mul(sub(fx1, s.ix), sub(fy1, s.iy));
  t.wne = mul(sub(s.ix, fx0), sub(fy1, s.iy));
  t.wsw = mul(sub(fx1, s.ix), sub(s.iy, fy0));
  t.wse = mul(sub(s.ix, fx0), sub(s.iy, fy0));
  const bool xin = (s.x0 + 1) < W, yin = (s.y0 + 1) < H;
  t.bne = xin;
  t.bsw = yin;
  t.bse = xin && yin;
  t.onw = s.y0 * W + s.x0;
  t.one = t.onw + (xin ? 1 : 0);
  t.osw = t.onw + (yin ? W : 0);
  t.ose = t.osw + (xin ? 1 : 0);
}

BBD_HD float tap_channel(const float* plane, const Taps& t) {
  float acc = mul(plane[t.onw], t.wnw);
  if (t.bne) acc = fma_(plane[t.one], t.wne, acc);
  if (t.bsw) acc = fma_(plane[t.osw], t.wsw, acc);
  if (t.bse) acc = fma_(plane[t.ose], t.wse, acc);
  return acc;
}

// d(sampled value)/d(ix, iy) of one channel, to be scaled by the upstream gradient
// (ATen grid_sampler_2d_backward, bilinear).  Out-of-range taps read as absent.
BBD_HD void tap_channel_grad(const float* plane, const Sample& s, const Taps& t, float g, float& gix, float& giy) {
  const float fx0 = (float)s.x0, fy0 = (float)s.y0;
  const float fx1 = fx0 + 1.0f, fy1 = fy0 + 1.0f;
  const float ex1 = sub(fx1, s.ix), ex0 = sub(s.ix, fx0);
  const float ey1 = sub(fy1, s.iy), ey0 = sub(s.iy, fy0);
  const float vnw = plane[t.onw];
  gix -= vnw * ey1 * g;
  giy -= vnw * ex1 * g;
  if (t.bne) { const float v = plane[t.one]; gix += v * ey1 * g; giy -= v * ex0 * g; }
  if (t.bsw) { const float v = plane[t.osw]; gix -= v * ey0 * g; giy += v * ex1 * g; }
  if (t.bse) { const float v = plane[t.ose]; gix += v * ey0 * g; giy += v * ex0 * g; }
}

// Chain (gix, giy) = dL/d(source coords) back to the depth of the pixel and to P.
// Unnormalise o normalise is the identity on the projected pixel, so d ix / d ux = 1
// (times the clip mask).  ux = cx / zz, uy = cy / zz.
BBD_HD void chain_to_depth_pose(const Cam& c, const Sample& s, float gix, float giy, float& gdepth, float gP[12]) {
  const float gux = gix * s.mx, guy = giy * s.my;
  const float inv = rcp_approx(s.zz);
  const float gcx = gux * inv, gcy = guy * inv;
  const float gcz = -(gux * s.ux + guy * s.uy) * inv;
  gP[0] += gcx * s.X; gP[1] += gcx * s.Y; gP[2] += gcx * s.Z; gP[3] += gcx;
  gP[4] += gcy * s.X; gP[5] += gcy * s.Y; gP[6] += gcy * s.Z; gP[7] += gcy;
  gP[8] += gcz * s.X; gP[9] += gcz * s.Y; gP[10] += gcz * s.Z; gP[11] += gcz;
  const float gX = c.p[0] * gcx + c.p[4] * gcy + c.p[8] * gcz;
  const float gY = c.p[1] * gcx + c.p[5] * gcy + c.p[9] * gcz;
  const float gZ = c.p[2] * gcx + c.p[6] * gcy + c.p[10] * gcz;
  gdepth += gX * s.rx + gY * s.ry + gZ * s.rz;
}

// ---- SSIM (layers.py:235-249) ----------------------------------------------
// Window sums are accumulated row-major like ATen's avg_pool2d and divided by 9.
struct WinX {  // per-channel window sums involving the warped image
  float sx, sxx, sxy;
};
struct WinY {  // per-channel target statistics: mean and variance term
  float mu, sig;
};

BBD_HD float ninth(float s) { return div_const(s, 9.0f, 0.111111111938953399658203125f); }

BBD_HD WinY target_stats(float sy, float syy) {
  WinY w;
  w.mu = ninth(sy);
  w.sig = sub(ninth(syy), mul(w.mu, w.mu));
  return w;
}

// One channel of SSIM's clamped dissimilarity; also returns the pieces the backward needs.
struct SsimParts {
  float mux, sigx, sigxy, n1, n2, d1, d2, r, raw;
};

// ... from the window moments (mean, variance term, covariance term) of the warped image
BBD_HD float ssim_from_moments(float mux, float sigx, float sigxy, const WinY& wy, SsimParts& q);

BBD_HD float ssim_channel(const WinX& wx, const WinY& wy, SsimParts& q) {
  const float mux = ninth(wx.sx);
  const float sigx = sub(ninth(wx.sxx), mul(mux, mux));
  const float sigxy = sub(ninth(wx.sxy), mul(mux, wy.mu));
  return ssim_from_moments(mux, sigx, sigxy, wy, q);
}

BBD_HD float ssim_from_moments(float mux, float sigx, float sigxy, const WinY& wy, SsimParts& q) {
  q.mux = mux;
  q.sigx = sigx;
  q.sigxy = sigxy;
  q.n1 = add(mul(mul(2.0f, q.mux), wy.mu), BBD_C1);
  q.n2 = add(mul(2.0f, q.sigxy), BBD_C2);
  q.d1 = add(add(mul(q.mux, q.mux), mul(wy.mu, wy.mu)), BBD_C1);
  q.d2 = add(add(q.sigx, wy.sig), BBD_C2);
  q.r = div_(mul(q.n1, q.n2), mul(q.d1, q.d2));
  q.raw = mul(sub(1.0f, q.r), 0.5f);
  return fminf(fmaxf(q.raw, 0.0f), 1.0f);
}

// Two window centres at once (same operation order, hence bit-identical to ssim_channel).
BBD_HD f2 ninth(const f2& s) { return div_const(s, 9.0f, 0.111111111938953399658203125f); }
// (also hands back the window moments, which is what the winner selection keeps for the backward)
struct SsimParts2 {
  f2 mux, sigx, sigxy, n1, n2, d1, d2, r, raw;
};
BBD_HD f2 ssim_from_moments2(const f2& mux, const f2& sigx, const f2& sigxy, const f2& muy, const f2& sigy, SsimParts2& q) {
  q.mux = mux;
  q.sigx = sigx;
  q.sigxy = sigxy;
  q.n1 = add(mul(mul(bc2(2.0f), mux), muy), bc2(BBD_C1));
  q.n2 = add(mul(bc2(2.0f), sigxy), bc2(BBD_C2));
  q.d1 = add(add(mul(mux, mux), mul(muy, muy)), bc2(BBD_C1));
  q.d2 = add(add(sigx, sigy), bc2(BBD_C2));
  q.r = div_(mul(q.n1, q.n2), mul(q.d1, q.d2));
  q.raw = mul(sub(bc2(1.0f), q.r), bc2(0.5f));
  return mk2(fminf(fmaxf(q.raw.x, 0.0f), 1.0f), fminf(fmaxf(q.raw.y, 0.0f), 1.0f));
}
BBD_HD f2 ssim_channel2(const f2& sx, const f2& sxx, const f2& sxy, const f2& muy, const f2& sigy, f2& mux, f2& sigx,
                        f2& sigxy) {
  mux = ninth(sx);
  sigx = sub(ninth(sxx), mul(mux, mux));
  sigxy = sub(ninth(sxy), mul(mux, muy));
  SsimParts2 q;
  return ssim_from_moments2(mux, sigx, sigxy, muy, sigy, q);
}

// Coefficients (a, b, c) such that d(value)/d x(u) = a + b*x(u) + c*y(u) for every pixel u of
// the window, `g` being the upstream gradient of the clamped value.  torch.clamp passes the
// gradient on the closed interval [0,1].
BBD_HD void ssim_coefs(const SsimParts& q, const WinY& wy, float g, float& a, float& b, float& c) {
  if (!(q.raw >= 0.0f && q.raw <= 1.0f)) { a = b = c = 0.0f; return; }
  const float gr = -0.5f * g;                  // raw = (1 - r)/2
  const float invd = rcp_approx(q.d1 * q.d2);
  const float r_n = invd;                      // dr/dn
  const float r_d = -q.r * invd;               // dr/dd
  const float r_sigxy = r_n * q.n1 * 2.0f;
  const float r_sigx = r_d * q.d1;
  const float r_mux = r_n * q.n2 * 2.0f * wy.mu + r_d * q.d2 * 2.0f * q.mux  // direct
                      - 2.0f * q.mux * r_sigx - wy.mu * r_sigxy;           // through sigma_x, sigma_xy
  const float k = gr * (1.0f / 9.0f);
  a = k * r_mux;
  b = k * 2.0f * r_sigx;
  c = k * r_sigxy;
}

// ssim_coefs for two channels at once (gradient-only arithmetic, packed)
BBD_HD void ssim_coefs2(const SsimParts2& q, const f2& muy, float g, f2& a, f2& b, f2& c) {
  const f2 gr = bc2(-0.5f * g);
  const f2 den = mul(q.d1, q.d2);
  const f2 invd = mk2(rcp_approx(den.x), rcp_approx(den.y));
  const f2 two = bc2(2.0f);
  const f2 r_d = mul(sub(bc2(0.0f), q.r), invd);
  const f2 r_sigxy = mul(mul(invd, q.n1), two);
  const f2 r_sigx = mul(r_d, q.d1);
  // direct terms, then the paths through sigma_x and sigma_xy
  f2 r_mux = fma_(mul(mul(invd, q.n2), two), muy, mul(mul(mul(r_d, q.d2), two), q.mux));
  r_mux = sub(r_mux, fma_(mul(two, q.mux), r_sigx, mul(muy, r_sigxy)));
  const f2 k = mul(gr, bc2(1.0f / 9.0f));
  a = mul(k, r_mux);
  b = mul(mul(k, two), r_sigx);
  c = mul(k, r_sigxy);
  if (!(q.raw.x >= 0.0f && q.raw.x <= 1.0f)) { a.x = b.x = c.x = 0.0f; }
  if (!(q.raw.y >= 0.0f && q.raw.y <= 1.0f)) { a.y = b.y = c.y = 0.0f; }
}

// Same for the target image: d(value)/d y(u) = a + b*y(u) + c*x(u)   (used by the SSIM operator).
BBD_HD void ssim_coefs_y(const SsimParts& q, const WinY& wy, float g, float& a, float& b, float& c) {
  if (!(q.raw >= 0.0f && q.raw <= 1.0f)) { a = b = c = 0.0f; return; }
  const float gr = -0.5f * g;
  const float invd = rcp_approx(q.d1 * q.d2);
  const float r_n = invd, r_d = -q.r * invd;
  const float r_sigxy = r_n * q.n1 * 2.0f;
  const float r_sigy = r_d * q.d1;
  const float r_muy = r_n * q.n2 * 2.0f * q.mux + r_d * q.d2 * 2.0f * wy.mu - 2.0f * wy.mu * r_sigy - q.mux * r_sigxy;
  const float k = gr * (1.0f / 9.0f);
  a = k * r_muy;
  b = k * 2.0f * r_sigy;
  c = k * r_sigxy;
}

// 0.85 * mean_c(ssim) + 0.15 * mean_c(l1)   (trainer.py:478-485); channel mean = sum * (1/3).
BBD_HD float photometric_mix(float ssim_sum, float l1_sum, bool no_ssim) {
  const float l1 = mul(l1_sum, BBD_THIRD);
  if (no_ssim) return l1;
  return add(mul(BBD_W_SSIM, mul(ssim_sum, BBD_THIRD)), mul(BBD_W_L1, l1));
}

}  // namespace bbd
