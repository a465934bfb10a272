// fsr_kernels.cuh -- FSR1 EASU (upscale) and RCAS (sharpen) for sm_100a.
//
// Replaces the two D3D11 compute dispatches of the reference:
//   g_FSRUpscaleShader = src/fsr/fsr_easu.hlsl:38-64 -> FsrEasuF, src/fsr/ffx_fsr1.h:315-437
//   g_FSRSharpenShader = src/fsr/fsr_rcas.hlsl:29-55 -> FsrRcasF, src/fsr/ffx_fsr1.h:684-769
// (citations relative to /root/reference/).  Not a translation of the HLSL: the work is
// re-tiled for a CTA of 8 warps over a 64x32 output tile,
//   * the source tile (+halo) is decoded ONCE per texel into shared memory (float4 rgb + luma);
//     the reference decodes every texel ~21 times through 36 Gather4s per pixel,
//   * EASU's direction/length analysis (FsrEasuSetF) depends only on the '+' neighbourhood of a
//     SOURCE texel, so it is evaluated once per source texel into a shared feature tile and
//     each output pixel bilinearly blends four float4 features instead of redoing 4 x ~25 ops,
//   * one warp owns one 16x16 output group, so the reference's per-workgroup radius test is a
//     warp-uniform branch (no divergence) with the bilinear / copy fast path fused in.
// Arithmetic order inside each reference function is kept where kStrict is set, so the strict
// build is bit-identical to the reference lines; the fast build regroups the 12 tap offsets
// (v = A*o - A*pp for integer o) and lets ptxas contract FMAs.
#pragma once

#include "device_common.cuh"
#include "tma_utils.cuh"

namespace ovrfsr {
inline namespace OVRFSR_MODE_NS {

constexpr int kTileW = 64;   // output tile of one CTA
constexpr int kTileH = 32;
constexpr int kThreads = 256; // 8 warps, one per 16x16 group

struct EasuArgs {
  ImageRO src;
  ImageRW dst;
  float c0x, c0y, c0z, c0w; // const0 of FsrEasuCon: out->in scale and offset
  uint32_t centre[4];
  uint32_t radiusSq;
  float radW, radH;         // (float)Radius.z, (float)Radius.w for Bilinear()
  int tileW, tileH;         // shared source tile extent in texels
  // When RCAS follows in the same apply (ctx path only): outside-radius groups are final after this pass -- RCAS would
  // only copy them (x the debug tint) -- so they are written straight to the final image `direct`, and to the
  // intermediate `dst` only where an edge-adjacent group is inside the radius (RCAS reads one pixel across the edge).
  ImageRW direct;           // ptr == nullptr: plain dispatch
  float tintGB;             // 1 - debug*0.3 of the following RCAS pass
  int x0, y0;               // src's origin in the texture srcMap describes (0, 0 unless src is a rectangle of it)
};

struct RcasArgs {
  ImageRO src;
  ImageRW dst;
  float sharp;              // const0[0] as float
  float tintGB;             // 1 - debug*0.3 (fsr_rcas.hlsl:46)
  uint32_t centre[4];
  uint32_t radiusSq;
  int skipOutside;          // the preceding EASU launch already wrote the outside-radius groups to dst (EasuArgs::direct)
  int opaqueSrc;            // B8G8R8X8 source: the X byte reads as alpha 1 (only the outside-radius copy looks at alpha)
  // TMA variant: src is the rectangle at (x0, y0) of the texture srcMap describes.  Tile boxes start at x = ox0 + boxX
  // (boxX = floor4(x0 - 1), a multiple of 4: the tile's first texel x0 - 1 lies boxShift = x0 - 1 - boxX texels into
  // the box) and y = oy0 - 1 + y0.  zeroOutside: the rectangle is smaller than the texture, so the texels a box holds
  // outside it are real data the kernel must replace by Texture2D.Load's out-of-bounds zero.
  int y0, boxX, boxShift, zeroOutside;
};

// out pixel -> source position; the same instruction sequence is used for the tile origin and
// for every pixel so that both agree to the bit.
__device__ __forceinline__ float easu_pos(int p, float scale, float offs) { return mul_add_unfused((float)p, scale, offs); }

// FsrEasuSetF (ffx_fsr1.h:275-313) minus the bilinear weight: the per-source-texel part.
//   a
// b c d      returns (dirX, dirY, lenX, lenY)
//   e
__device__ __forceinline__ float4 easu_feature(float lA, float lB, float lC, float lD, float lE) {
  const float dc = lD - lC, cb = lC - lB;
  float lenX = prx_lo_rcp(fmaxf(fabsf(dc), fabsf(cb)));
  const float dirX = lD - lB;
  lenX = __saturatef(fabsf(dirX) * lenX);
  lenX *= lenX;
  const float ec = lE - lC, ca = lC - lA;
  float lenY = prx_lo_rcp(fmaxf(fabsf(ec), fabsf(ca)));
  const float dirY = lE - lA;
  lenY = __saturatef(fabsf(dirY) * lenY);
  lenY *= lenY;
  return make_float4(dirX, dirY, lenX, lenY);
}

// ---- strict math: FsrEasuF in the reference's operation order (scalar) ----------------------------------------
// (A two-lane FMUL2/FADD2 version exists in the history: it is bit-exact too -- with the neutral-element trick of
// device_common.cuh against ptxas' f32x2 contraction -- but every strict mul and add is its own FMA-pipe op either
// way, so it was FMA-pipe-bound and 3 % slower than this scalar form.)
// Products the reference recomputes per tap are formed once: off.x*dir.x and off.x*(-dir.y) for the 4 distinct
// off.x, off.y*dir.y and off.y*dir.x for the 4 distinct off.y -- same operands, same product, 16 multiplies
// instead of 48.
// FsrEasuTapF, ffx_fsr1.h:239-272, from the two products of each coordinate
__device__ __forceinline__ void easu_tap_ref(float &aR, float &aG, float &aB, float &aW, float xdx, float ydy, float xndy,
                                             float ydx, float len0, float len1, float lob, float clp, const float4 c) {
  float vx = xdx + ydy;   // (off.x*dir.x) + (off.y*dir.y)
  float vy = xndy + ydx;  // (off.x*(-dir.y)) + (off.y*dir.x)
  vx *= len0;
  vy *= len1;
  float d2 = vx * vx + vy * vy;
  d2 = fminf(d2, clp);
  float wB = (float)(2.0 / 5.0) * d2 + (float)(-1.0);
  float wA = lob * d2 + (float)(-1.0);
  wB *= wB;
  wA *= wA;
  wB = (float)(25.0 / 16.0) * wB + (float)(-(25.0 / 16.0 - 1.0));
  const float w = wB * wA;
  aR += c.x * w; aG += c.y * w; aB += c.z * w;
  aW += w;
}

// FsrEasuF, ffx_fsr1.h:315-437, for the output pixel whose 'f' texel sits at tile coords (ix,iy)
// with sub-texel phase (ppx,ppy).  sC = decoded colours (xyz), sF = per-texel features.
template <int TW>
__device__ __forceinline__ float3 easu_filter(const float4 *__restrict__ sC, const float4 *__restrict__ sF, int ix, int iy,
                                              float ppx, float ppy) {
  // direction + length: bilinear blend of the four corner features (:380-386)
  const float4 *fr = sF + iy * TW + ix;
  const float4 Ff = fr[0], Fg = fr[1], Fj = fr[TW], Fk = fr[TW + 1];
  const float qx = 1.0f - ppx, qy = 1.0f - ppy;
  const float wf = qx * qy, wg = ppx * qy, wj = qx * ppy, wk = ppx * ppy;
  float dirX = 0.0f, dirY = 0.0f, len = 0.0f;
  dirX += Ff.x * wf; len += Ff.z * wf; dirY += Ff.y * wf; len += Ff.w * wf;
  dirX += Fg.x * wg; len += Fg.z * wg; dirY += Fg.y * wg; len += Fg.w * wg;
  dirX += Fj.x * wj; len += Fj.z * wj; dirY += Fj.y * wj; len += Fj.w * wj;
  dirX += Fk.x * wk; len += Fk.z * wk; dirY += Fk.y * wk; len += Fk.w * wk;

  // normalise (:389-395)
  const float dir2x = dirX * dirX, dir2y = dirY * dirY;
  float dirR = dir2x + dir2y;
  const bool zro = dirR < (float)(1.0 / 32768.0);
  dirR = prx_lo_rsq(dirR);
  dirR = zro ? 1.0f : dirR;
  dirX = zro ? 1.0f : dirX;
  dirX *= dirR;
  dirY *= dirR;
  // shape (:397-409)
  len = len * 0.5f;
  len *= len;
  const float stretch = (dirX * dirX + dirY * dirY) * prx_lo_rcp(fmaxf(fabsf(dirX), fabsf(dirY)));
  const float len0 = 1.0f + (stretch - 1.0f) * len;
  const float len1 = 1.0f + (-0.5f) * len;
  const float lob = 0.5f + (float)((1.0 / 4.0 - 0.04) - 0.5) * len;
  const float clp = prx_lo_rcp(lob);

  // the 4 distinct off.x / off.y values and their products with dir (shared by the 12 taps)
  const float ndirY = -dirY;
  const float ox0 = -1.0f - ppx, ox1 = 0.0f - ppx, ox2 = 1.0f - ppx, ox3 = 2.0f - ppx;
  const float oy0 = -1.0f - ppy, oy1 = 0.0f - ppy, oy2 = 1.0f - ppy, oy3 = 2.0f - ppy;
  const float xd0 = ox0 * dirX, xd1 = ox1 * dirX, xd2 = ox2 * dirX, xd3 = ox3 * dirX;
  const float xn0 = ox0 * ndirY, xn1 = ox1 * ndirY, xn2 = ox2 * ndirY, xn3 = ox3 * ndirY;
  const float yd0 = oy0 * dirY, yd1 = oy1 * dirY, yd2 = oy2 * dirY, yd3 = oy3 * dirY;
  const float yx0 = oy0 * dirX, yx1 = oy1 * dirX, yx2 = oy2 * dirX, yx3 = oy3 * dirX;

  //    b c
  //  e f g h
  //  i j k l
  //    n o
  const float4 *r0 = sC + (iy - 1) * TW + ix;
  const float4 f = r0[TW], g = r0[TW + 1], j = r0[2 * TW], k = r0[2 * TW + 1];
  float aR = 0.0f, aG = 0.0f, aB = 0.0f, aW = 0.0f;
  // reference accumulation order (:423-434): b c i j f e k l h g o n   (index 0..3 <-> offset -1..2)
  easu_tap_ref(aR, aG, aB, aW, xd1, yd0, xn1, yx0, len0, len1, lob, clp, r0[0]);          // b ( 0,-1)
  easu_tap_ref(aR, aG, aB, aW, xd2, yd0, xn2, yx0, len0, len1, lob, clp, r0[1]);          // c ( 1,-1)
  easu_tap_ref(aR, aG, aB, aW, xd0, yd2, xn0, yx2, len0, len1, lob, clp, r0[2 * TW - 1]); // i (-1, 1)
  easu_tap_ref(aR, aG, aB, aW, xd1, yd2, xn1, yx2, len0, len1, lob, clp, j);              // j ( 0, 1)
  easu_tap_ref(aR, aG, aB, aW, xd1, yd1, xn1, yx1, len0, len1, lob, clp, f);              // f ( 0, 0)
  easu_tap_ref(aR, aG, aB, aW, xd0, yd1, xn0, yx1, len0, len1, lob, clp, r0[TW - 1]);     // e (-1, 0)
  easu_tap_ref(aR, aG, aB, aW, xd2, yd2, xn2, yx2, len0, len1, lob, clp, k);              // k ( 1, 1)
  easu_tap_ref(aR, aG, aB, aW, xd3, yd2, xn3, yx2, len0, len1, lob, clp, r0[2 * TW + 2]); // l ( 2, 1)
  easu_tap_ref(aR, aG, aB, aW, xd3, yd1, xn3, yx1, len0, len1, lob, clp, r0[TW + 2]);     // h ( 2, 0)
  easu_tap_ref(aR, aG, aB, aW, xd2, yd1, xn2, yx1, len0, len1, lob, clp, g);              // g ( 1, 0)
  easu_tap_ref(aR, aG, aB, aW, xd2, yd3, xn2, yx3, len0, len1, lob, clp, r0[3 * TW + 1]); // o ( 1, 2)
  easu_tap_ref(aR, aG, aB, aW, xd1, yd3, xn1, yx3, len0, len1, lob, clp, r0[3 * TW]);     // n ( 0, 2)

  // min/max of the four nearest (:416-419), normalise and de-ring (:437)
  const float mnR = fminf(fminf(f.x, fminf(g.x, j.x)), k.x), mxR = fmaxf(fmaxf(f.x, fmaxf(g.x, j.x)), k.x);
  const float mnG = fminf(fminf(f.y, fminf(g.y, j.y)), k.y), mxG = fmaxf(fmaxf(f.y, fmaxf(g.y, j.y)), k.y);
  const float mnB = fminf(fminf(f.z, fminf(g.z, j.z)), k.z), mxB = fmaxf(fmaxf(f.z, fmaxf(g.z, j.z)), k.z);
  const float r = rcp_mode(aW);
  return make_float3(fminf(mxR, fmaxf(mnR, aR * r)), fminf(mxG, fmaxf(mnG, aG * r)), fminf(mxB, fmaxf(mnB, aB * r)));
}

// ---- fast math: FsrEasuF regrouped for the FP32x2 pipe ----------------------------------------------------
// Same function as easu_filter, evaluated differently (results differ from the reference lines in the last
// bits only; <= 1 LSB after RGBA8 rounding):
//   * the squared rotated/stretched tap distance is a quadratic form of the integer tap offset,
//       d2(ox,oy) = Q00*dx^2 + 2*Q01*dx*dy + Q11*dy^2,  dx = ox-ppx, dy = oy-ppy,  Q = M^T M,
//     so one FADD2 + one FFMA2 yield d2 for two horizontally adjacent taps (A_P + B_j, E_P*dy_j);
//   * the window polynomial is expanded: 25/16*(2/5 t-1)^2 - 9/16 = (t/4 - 5/4) t + 1;
//   * the colour tile stores (r,g,b,1): two FFMA2 per tap accumulate (r,g) and (b, weight) at once;
//   * feature blending, normalisation and setup are packed the same way.  ~100 packed + ~40 scalar FP
//     instructions per pixel instead of ~250 scalar ones.
__device__ __forceinline__ f2 easu_w2(f2 A, float B, f2 E, float dy, float clp, float lob) {
  f2 t = fma2(E, bc(dy), add2(A, bc(B)));
  t.x = fminf(t.x, clp);
  t.y = fminf(t.y, clp);
  const f2 base = fma2(fma2(t, bc(0.25f), bc(-1.25f)), t, bc(1.0f));
  f2 win = fma2(t, bc(lob), bc(-1.0f));
  win = mul2(win, win);
  return mul2(base, win);
}
__device__ __forceinline__ void easu_acc(f2 &aRG, f2 &aBW, const float4 c, float w) {
  aRG = fma2(make_float2(c.x, c.y), bc(w), aRG);
  aBW = fma2(make_float2(c.z, c.w), bc(w), aBW); // c.w == 1: the weight sum rides along
}

template <int TW>
__device__ __forceinline__ float3 easu_filter_fast(const float4 *__restrict__ sC, const float4 *__restrict__ sF, int ix,
                                                   int iy, float ppx, float ppy) {
  const float4 *fr = sF + iy * TW + ix;
  const float4 Ff = fr[0], Fg = fr[1], Fj = fr[TW], Fk = fr[TW + 1];
  const float qx = 1.0f - ppx, qy = 1.0f - ppy;
  const f2 wt = mul2(make_float2(qx, ppx), bc(qy)), wb = mul2(make_float2(qx, ppx), bc(ppy)); // (wf,wg) (wj,wk)
  f2 dir = mul2(make_float2(Ff.x, Ff.y), bc(wt.x));
  f2 ln = mul2(make_float2(Ff.z, Ff.w), bc(wt.x));
  dir = fma2(make_float2(Fg.x, Fg.y), bc(wt.y), dir); ln = fma2(make_float2(Fg.z, Fg.w), bc(wt.y), ln);
  dir = fma2(make_float2(Fj.x, Fj.y), bc(wb.x), dir); ln = fma2(make_float2(Fj.z, Fj.w), bc(wb.x), ln);
  dir = fma2(make_float2(Fk.x, Fk.y), bc(wb.y), dir); ln = fma2(make_float2(Fk.z, Fk.w), bc(wb.y), ln);
  float len = ln.x + ln.y;

  f2 dd = mul2(dir, dir);
  float dirR = dd.x + dd.y;
  const bool zro = dirR < (float)(1.0 / 32768.0);
  dirR = zro ? 1.0f : prx_lo_rsq(dirR);
  dir.x = zro ? 1.0f : dir.x;
  dir = mul2(dir, bc(dirR));
  len = len * 0.5f;
  len *= len;
  dd = mul2(dir, dir);
  const float stretch = (dd.x + dd.y) * prx_lo_rcp(fmaxf(fabsf(dir.x), fabsf(dir.y)));
  const float len0 = fmaf(stretch - 1.0f, len, 1.0f);
  const float len1 = fmaf(-0.5f, len, 1.0f);
  const float lob = fmaf((float)((1.0 / 4.0 - 0.04) - 0.5), len, 0.5f);
  const float clp = prx_lo_rcp(lob);

  // Q = M^T M with M = diag(len0,len1) * Rot(dir):  Q00 = dx^2 L0 + dy^2 L1, Q11 = dy^2 L0 + dx^2 L1, Q01 = dx dy (L0-L1)
  const float L0 = len0 * len0, L1 = len1 * len1;
  const float Q00 = fmaf(dd.x, L0, dd.y * L1), Q11 = fmaf(dd.y, L0, dd.x * L1);
  const float Q01x2 = 2.0f * (dir.x * dir.y) * (L0 - L1);
  // tap offsets: x pairs (-1,0) (0,1) (1,2), y scalars -1,0,1,2
  const f2 mpx = bc(-ppx), mpy = bc(-ppy);
  const f2 dxA = add2(make_float2(-1.0f, 0.0f), mpx), dxB = add2(make_float2(0.0f, 1.0f), mpx),
           dxC = add2(make_float2(1.0f, 2.0f), mpx);
  const f2 dyA = add2(make_float2(-1.0f, 0.0f), mpy), dyB = add2(make_float2(1.0f, 2.0f), mpy);
  const f2 qq = bc(Q00), ee = bc(Q01x2), q11 = bc(Q11);
  const f2 AA = mul2(mul2(dxA, dxA), qq), AB = mul2(mul2(dxB, dxB), qq), AC = mul2(mul2(dxC, dxC), qq);
  const f2 EA = mul2(dxA, ee), EB = mul2(dxB, ee), EC = mul2(dxC, ee);
  const f2 BA = mul2(mul2(dyA, dyA), q11), BB = mul2(mul2(dyB, dyB), q11); // (B_-1,B_0) (B_1,B_2)

  //    b c
  //  e f g h
  //  i j k l
  //    n o
  const float4 *r0 = sC + (iy - 1) * TW + ix;
  f2 aRG = bc(0.0f), aBW = bc(0.0f);
  {
    const float4 b = r0[0], c = r0[1];
    const f2 w = easu_w2(AB, BA.x, EB, dyA.x, clp, lob);
    easu_acc(aRG, aBW, b, w.x); easu_acc(aRG, aBW, c, w.y);
  }
  const float4 f = r0[TW], g = r0[TW + 1], j = r0[2 * TW], k = r0[2 * TW + 1];
  {
    const float4 e = r0[TW - 1], h = r0[TW + 2];
    const f2 w0 = easu_w2(AA, BA.y, EA, dyA.y, clp, lob), w1 = easu_w2(AC, BA.y, EC, dyA.y, clp, lob);
    easu_acc(aRG, aBW, e, w0.x); easu_acc(aRG, aBW, f, w0.y);
    easu_acc(aRG, aBW, g, w1.x); easu_acc(aRG, aBW, h, w1.y);
  }
  {
    const float4 i = r0[2 * TW - 1], l = r0[2 * TW + 2];
    const f2 w0 = easu_w2(AA, BB.x, EA, dyB.x, clp, lob), w1 = easu_w2(AC, BB.x, EC, dyB.x, clp, lob);
    easu_acc(aRG, aBW, i, w0.x); easu_acc(aRG, aBW, j, w0.y);
    easu_acc(aRG, aBW, k, w1.x); easu_acc(aRG, aBW, l, w1.y);
  }
  {
    const float4 n = r0[3 * TW], o = r0[3 * TW + 1];
    const f2 w = easu_w2(AB, BB.y, EB, dyB.y, clp, lob);
    easu_acc(aRG, aBW, n, w.x); easu_acc(aRG, aBW, o, w.y);
  }
  const float mnR = fminf(fminf(f.x, fminf(g.x, j.x)), k.x), mxR = fmaxf(fmaxf(f.x, fmaxf(g.x, j.x)), k.x);
  const float mnG = fminf(fminf(f.y, fminf(g.y, j.y)), k.y), mxG = fmaxf(fmaxf(f.y, fmaxf(g.y, j.y)), k.y);
  const float mnB = fminf(fminf(f.z, fminf(g.z, j.z)), k.z), mxB = fmaxf(fmaxf(f.z, fmaxf(g.z, j.z)), k.z);
  const float r = rcp_mode(aBW.y);
  return make_float3(fminf(mxR, fmaxf(mnR, aRG.x * r)), fminf(mxG, fmaxf(mnG, aRG.y * r)), fminf(mxB, fmaxf(mnB, aBW.x * r)));
}

// Bilinear(), fsr_easu.hlsl:33-36: SampleLevel(linearClamp, float2(pos)/Radius.zw) -- no half-texel
// offset; coordinates snapped to 1/256 texel like D3D11's fixed-point sampler.  The sample position is separable:
// the x part (one IEEE divide, snap, floor) depends only on the output column and the y part only on the output row,
// so each is evaluated once per column / row instead of once per pixel -- same operations, same bits.
struct BilinAxis { int t0, t1; float f; }; // clamped tile coordinates of the two taps and the weight of the second
__device__ __forceinline__ BilinAxis easu_bilinear_axis(int p, float rad, int srcExtent, int tileOrigin, int tileExtent) {
  const float u = (float)p / rad;
  const float s = snap_subtexel(mul_add_unfused(u, (float)srcExtent, -0.5f));
  const float s0 = floorf(s);
  BilinAxis r;
  r.f = s - s0;
  r.t0 = clampi((int)s0 - tileOrigin, 0, tileExtent - 1);
  r.t1 = clampi((int)s0 + 1 - tileOrigin, 0, tileExtent - 1);
  return r;
}
__device__ __forceinline__ float3 easu_bilinear(const float4 *__restrict__ sC, int tw, const BilinAxis ax, const BilinAxis ay) {
  const float4 c00 = sC[ay.t0 * tw + ax.t0], c10 = sC[ay.t0 * tw + ax.t1];
  const float4 c01 = sC[ay.t1 * tw + ax.t0], c11 = sC[ay.t1 * tw + ax.t1];
  const float fx = ax.f, fy = ay.f, wx0 = 1.0f - fx, wy0 = 1.0f - fy;
  const float tR = c00.x * wx0 + c10.x * fx, bR = c01.x * wx0 + c11.x * fx;
  const float tG = c00.y * wx0 + c10.y * fx, bG = c01.y * wx0 + c11.y * fx;
  const float tB = c00.z * wx0 + c10.z * fx, bB = c01.z * wx0 + c11.z * fx;
  return make_float3(tR * wy0 + bR * fy, tG * wy0 + bG * fy, tB * wy0 + bB * fy);
}

// 3-channel decode of a packed RGBA8/BGRA8 texel (EASU never reads source alpha: its output alpha is 1).
// ALWAYS the exact decode, also in fast math: where luma is flat but chroma varies, FsrEasuSetF divides rounding
// noise by rounding noise (|lD-lB| / max(|lD-lC|,|lC-lB|) with all three lumas equal up to the last bit), so the
// edge strength there is defined by the exact bits of the decoded values; a decode that is 1 ulp off changes the
// result by several LSB at such pixels.
template <int FMT>
__device__ __forceinline__ float4 decode_rgb1(uint32_t p) {
  if constexpr (FMT == OVRFSR_FORMAT_RGB10A2) return make_float4(unorm10(p & 1023u), unorm10((p >> 10) & 1023u), unorm10((p >> 20) & 1023u), 1.0f);
  const float c0 = unorm8(byte_to_float<0>(p)), c1 = unorm8(byte_to_float<1>(p)), c2 = unorm8(byte_to_float<2>(p));
  if constexpr (FMT == OVRFSR_FORMAT_BGRA8) return make_float4(c2, c1, c0, 1.0f);
  return make_float4(c0, c1, c2, 1.0f);
}
template <int FMT>
__device__ __forceinline__ float4 decode_rgba(uint32_t p) {
  if constexpr (FMT == OVRFSR_FORMAT_RGB10A2) return decode_rgb10a2(p);
  const float c0 = byte_to_unorm_mode<0>(p), c1 = byte_to_unorm_mode<1>(p);
  const float c2 = byte_to_unorm_mode<2>(p), c3 = byte_to_unorm_mode<3>(p);
  if constexpr (FMT == OVRFSR_FORMAT_BGRA8) return make_float4(c2, c1, c0, c3);
  return make_float4(c0, c1, c2, c3);
}

// FLOAT -> intermediate UNORM -> FLOAT, the store / Load round trip of the two-dispatch form
template <int FMID>
__device__ __forceinline__ float4 mid_roundtrip(float r, float g, float b) {
  if constexpr (FMID == OVRFSR_FORMAT_RGB10A2) {
    return make_float4(unorm10(to_unorm<1023>(r)), unorm10(to_unorm<1023>(g)), unorm10(to_unorm<1023>(b)), 1.0f);
  } else {
    // to_unorm8 then the decode rcas_kernel applies to an RGBA8 source (decode_rgba: exact in strict math, the
    // single-FFMA form in fast math); the code is already an integer, so 2^23 + v is one LOP3 instead of a PRMT
    const uint32_t cr = to_unorm8(r) | 0x4B000000u, cg = to_unorm8(g) | 0x4B000000u, cb = to_unorm8(b) | 0x4B000000u;
    if constexpr (kStrict) {
      return make_float4(unorm8(u2f(cr) - 8388608.0f), unorm8(u2f(cg) - 8388608.0f), unorm8(u2f(cb) - 8388608.0f), 1.0f);
    } else {
      const float k = 1.0f / 255.0f;
      return make_float4(__fmaf_rn(u2f(cr), k, -8388608.0f * k), __fmaf_rn(u2f(cg), k, -8388608.0f * k),
                         __fmaf_rn(u2f(cb), k, -8388608.0f * k), 1.0f);
    }
  }
}

// TW  = shared tile row stride in texels (compile time, so every tap is base + immediate): 60 covers out->in
//       scales up to 0.81 for a 64-wide output tile (60 texels incl. the 4 TMA alignment columns), 72 the rest up to 1.0.
// TMA = the raw RGBA8 source box (tile + halo) arrives by cp.async.bulk.tensor into a double-buffered landing zone
//       and is decoded from there; otherwise (FP16/FP32 sources, unaligned pitch) texels are fetched with plain loads.
// Persistent: the grid is (CTAs per SM) x (SM count); each CTA walks tiles t = blockIdx.x, +gridDim.x, ... in
// row-major order and, in the TMA variant, has the NEXT tile's box in flight while it works on the current one.
constexpr int kEasuRowsPerThread = 5;  // tile rows handled by one warp: ceil(37 / 8)
constexpr int kEasuColsPerThread = 3;  // 32-wide column blocks: ceil(72 / 32)

// PAIRED = RCAS follows in the same apply (EasuArgs::direct is set): a compile-time variant, so that the plain dispatch
// keeps exactly the instruction stream it had without the pairing.
template <int FIN, int FOUT, int TW, bool TMA, bool PAIRED>
__global__ void __launch_bounds__(kThreads, 3) easu_kernel(const __grid_constant__ EasuArgs a,
                                                           const __grid_constant__ CUtensorMap srcMap) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ uint64_t tileBar;
  __shared__ BilinAxis sRowAxis[kTileH]; // Bilinear()'s row terms of this tile (outside-radius groups only)
  const int th = a.tileH, tn = TW * th;
  float4 *sC = reinterpret_cast<float4 *>(smem_raw);  // decoded colour (r,g,b,1)
  float4 *sF = sC + tn;                               // (dirX, dirY, lenX, lenY) per texel
  float *sL = reinterpret_cast<float *>(sF + tn);     // luma*2 plane (conflict-free stencil reads)
  const int rawW = a.tileW + 4;                       // TMA box width (origin floored to 4 texels)
  uint32_t *sRaw = reinterpret_cast<uint32_t *>(smem_raw + ((tn * 36 + 127) & ~127)); // landing zone (TMA only), 128-byte aligned

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tilesX = (a.dst.w + kTileW - 1) / kTileW, tilesY = (a.dst.h + kTileH - 1) / kTileH;
  const int numTiles = tilesX * tilesY;

  auto tile_origin = [&](int t, int &ox0, int &oy0, int &sx0, int &sy0) {
    const int ty = t / tilesX, tx = t - ty * tilesX;
    ox0 = tx * kTileW; oy0 = ty * kTileH;
    // source tile origin: one texel left/above the 'f' texel of the tile's first pixel
    sx0 = (int)floorf(easu_pos(ox0, a.c0x, a.c0z)) - 1;
    sy0 = (int)floorf(easu_pos(oy0, a.c0y, a.c0w)) - 1;
  };

  // Static schedule t = blockIdx.x, += gridDim.x.  (Taking tiles by cluster launch control, as nis_scaler_kernel does,
  // was measured too: 108.4 vs 106.9 us at radius 2.0 where all tiles cost the same, 56.0 vs 57.1 us at radius 0.5 --
  // not worth the extra latency on the tile loop here; profiles/r2_rejected_experiments.md.)
  int t = blockIdx.x;
  if constexpr (TMA) {
    if (tid == 0) {
      mbar_init(&tileBar, 1);
      fence_barrier_init();
      if (t < numTiles) {
        int ox0, oy0, sx0, sy0;
        tile_origin(t, ox0, oy0, sx0, sy0);
        mbar_arrive_expect_tx(&tileBar, (uint32_t)(rawW * th * 4));
        tma_load_2d(sRaw, &srcMap, (sx0 + a.x0) & ~3, sy0 + a.y0, &tileBar); // box origin 16-byte aligned in x
      }
    }
    __syncthreads();
  }

  uint32_t phase = 0;
  for (; t < numTiles; t += gridDim.x) {
    int ox0, oy0, sx0, sy0;
    tile_origin(t, ox0, oy0, sx0, sy0);
    // float-tile origin and width in source texels: the TMA variant keeps the box's aligned origin (aligned in the
    // texture, so within a rectangle at x0 % 4 != 0 it is up to 3 texels left of sx0)
    const int tx0 = TMA ? ((sx0 + a.x0) & ~3) - a.x0 : sx0;
    const int cols = TMA ? rawW : a.tileW;

    // this warp's 16x16 group and its radius test (warp-uniform)
    const uint32_t ggx = (uint32_t)(ox0 >> 4) + (warp & 3), ggy = (uint32_t)(oy0 >> 4) + (warp >> 2);
    const bool inside = group_inside(ggx * 16u + 8u, ggy * 16u + 8u, a.centre, a.radiusSq);

    // ---- stage 1: decode the clamped source tile once, loads batched per thread for ILP -------------
    if constexpr (TMA) {
      mbar_wait(&tileBar, phase); // this tile's box has landed (zeros outside the texture)
      phase ^= 1u;
      const uint32_t *raw = sRaw;
#pragma unroll
      for (int i = 0; i < kEasuColsPerThread; ++i) {
        const int tx = lane + 32 * i;
        if (tx < cols) {
          // clamp-to-edge: re-read the edge column / row of the image (of the rectangle: texels outside it are never used)
          const int rcol = clampi(tx0 + tx, 0, a.src.w - 1) - tx0;
          uint32_t px[kEasuRowsPerThread];
#pragma unroll
          for (int j = 0; j < kEasuRowsPerThread; ++j) {
            const int ty = warp + 8 * j;
            px[j] = ty < th ? raw[(clampi(sy0 + ty, 0, a.src.h - 1) - sy0) * rawW + rcol] : 0u;
          }
#pragma unroll
          for (int j = 0; j < kEasuRowsPerThread; ++j) {
            const int ty = warp + 8 * j;
            if (ty < th) {
              const float4 c = decode_rgb1<FIN>(px[j]);
              sL[ty * TW + tx] = c.z * 0.5f + (c.x * 0.5f + c.y); // luma*2, ffx_fsr1.h:363 (x0.5 exact: FMA-safe)
              sC[ty * TW + tx] = c;
            }
          }
        }
      }
    } else {
      // plain loads (FP16 / FP32 sources, unaligned pitch): a flat index over the tile, four texels per thread in
      // flight (no prefetch hides this latency, unlike the TMA variant)
      const int nTex = cols * th;
      const uint32_t colsRcp = 0xFFFFFFFFu / (uint32_t)cols + 1u; // ceil(2^32 / cols): q / cols == umulhi(q, colsRcp) for q < 2^32 / cols
#pragma unroll 4
      for (int q = tid; q < nTex; q += kThreads) {
        const int ty = (int)__umulhi((uint32_t)q, colsRcp), tx = q - ty * cols;
        const int gy = clampi(sy0 + ty, 0, a.src.h - 1), gx = clampi(tx0 + tx, 0, a.src.w - 1);
        float4 c = fetch_texel<FIN>(a.src.ptr + (size_t)gy * a.src.pitch, gx);
        sL[ty * TW + tx] = c.z * 0.5f + (c.x * 0.5f + c.y);
        c.w = 1.0f; // EASU ignores source alpha; the fast path accumulates the tap weight through this lane
        sC[ty * TW + tx] = c;
      }
    }
    // one row term per output row of the tile for the bilinear fallback (skipped when every group is inside)
    if (tid < kTileH && oy0 + tid < a.dst.h) sRowAxis[tid] = easu_bilinear_axis(oy0 + tid, a.radH, a.src.h, sy0, th);
    const int anyInside = __syncthreads_or(inside);
    const int tn2 = t + gridDim.x;
    if constexpr (TMA) {
      // the landing zone is fully decoded: refill it with the NEXT tile's box while this tile is filtered
      if (tid == 0 && tn2 < numTiles) {
        int nox, noy, nsx, nsy;
        tile_origin(tn2, nox, noy, nsx, nsy);
        fence_proxy_async();
        mbar_arrive_expect_tx(&tileBar, (uint32_t)(rawW * th * 4));
        tma_load_2d(sRaw, &srcMap, (nsx + a.x0) & ~3, nsy + a.y0, &tileBar);
      }
    }

    // ---- stage 2: per-source-texel direction/length features (only where EASU will run) -----------
    if (anyInside) {
#pragma unroll
      for (int i = 0; i < kEasuColsPerThread; ++i) {
        const int tx = 1 + lane + 32 * i;
        if (tx < cols - 1) {
          float lA[kEasuRowsPerThread], lB[kEasuRowsPerThread], lC[kEasuRowsPerThread], lD[kEasuRowsPerThread],
              lE[kEasuRowsPerThread];
#pragma unroll
          for (int j = 0; j < kEasuRowsPerThread; ++j) {
            const int ty = 1 + warp + 8 * j;
            if (ty < th - 1) {
              const float *l = sL + ty * TW + tx;
              lA[j] = l[-TW]; lB[j] = l[-1]; lC[j] = l[0]; lD[j] = l[1]; lE[j] = l[TW];
            }
          }
#pragma unroll
          for (int j = 0; j < kEasuRowsPerThread; ++j) {
            const int ty = 1 + warp + 8 * j;
            if (ty < th - 1) sF[ty * TW + tx] = easu_feature(lA[j], lB[j], lC[j], lD[j], lE[j]);
          }
        }
      }
      __syncthreads();
    }

    // ---- stage 3: one warp per 16x16 group, 8 pixels per lane --------------------------------------
    const int x = (int)ggx * 16 + (lane & 15);
    if (x < a.dst.w) {
      const int yFirst = (int)ggy * 16 + (lane >> 4);
      if (inside) {
        const float ppx_full = easu_pos(x, a.c0x, a.c0z);
        const float fpx = floorf(ppx_full);
        const float ppx = ppx_full - fpx;
        const int ix = (int)fpx - tx0;
#pragma unroll 2
        for (int k = 0; k < 8; ++k) {
          const int y = yFirst + 2 * k;
          if (y >= a.dst.h) break;
          const float ppy_full = easu_pos(y, a.c0y, a.c0w);
          const float fpy = floorf(ppy_full);
          float3 c;
          if constexpr (kStrict) c = easu_filter<TW>(sC, sF, ix, (int)fpy - sy0, ppx, ppy_full - fpy);
          else c = easu_filter_fast<TW>(sC, sF, ix, (int)fpy - sy0, ppx, ppy_full - fpy);
          store_opaque<FOUT>(a.dst.ptr + (size_t)y * a.dst.pitch, x, c.x, c.y, c.z);
        }
      } else {
        const BilinAxis ax = easu_bilinear_axis(x, a.radW, a.src.w, tx0, cols);
        constexpr bool direct = PAIRED && (FOUT == OVRFSR_FORMAT_RGBA8 || FOUT == OVRFSR_FORMAT_RGB10A2);
        // the intermediate is still needed where RCAS of an edge-adjacent inside group reads across the group edge
        const bool mid = !direct || group_inside(ggx * 16u - 8u, ggy * 16u + 8u, a.centre, a.radiusSq) ||
                         group_inside(ggx * 16u + 24u, ggy * 16u + 8u, a.centre, a.radiusSq) ||
                         group_inside(ggx * 16u + 8u, ggy * 16u - 8u, a.centre, a.radiusSq) ||
                         group_inside(ggx * 16u + 8u, ggy * 16u + 24u, a.centre, a.radiusSq);
#pragma unroll 2
        for (int k = 0; k < 8; ++k) {
          const int y = yFirst + 2 * k;
          if (y >= a.dst.h) break;
          const float3 c = easu_bilinear(sC, TW, ax, sRowAxis[y - oy0]);
          if (mid) store_opaque<FOUT>(a.dst.ptr + (size_t)y * a.dst.pitch, x, c.x, c.y, c.z);
          if constexpr (direct) {
            {
              uint8_t *row = a.direct.ptr + (size_t)y * a.direct.pitch;
              if (a.tintGB == 1.0f) {
                // RCAS's copy is the identity on UNORM codes (decode -> x1 -> encode): the same bits go to the final image
                store_opaque<FOUT>(row, x, c.x, c.y, c.z);
              } else {
                // OutputTexture[p] = mul * InputTexture[p] on the stored-then-loaded value (fsr_rcas.hlsl:45-53)
                const float4 m = mid_roundtrip<FOUT>(c.x, c.y, c.z);
                store_texel<FOUT>(row, x, 1.0f * m.x, a.tintGB * m.y, a.tintGB * m.z, 1.0f * m.w);
              }
            }
          }
        }
      }
    }
    __syncthreads(); // every warp is done with this tile before the next decode overwrites it
  }
}

// ------------------------------------------------------------------------------------------------
// RCAS
// ------------------------------------------------------------------------------------------------
constexpr int kRcasTW = kTileW + 4;  // float tile: 1-texel halo each side, padded to a multiple of 4 texels
constexpr int kRcasTH = kTileH + 2;
constexpr int kRcasRawW = kTileW + 8; // TMA box: starts 4 texels left of the tile (16-byte aligned origin), 1 used right

// FsrRcasF, ffx_fsr1.h:684-769 (FSR_RCAS_DENOISE / PASSTHROUGH_ALPHA undefined: fsr_rcas.hlsl:1-4), reference order
template <bool U8>
__device__ __forceinline__ float3 rcas_filter(const float4 b, const float4 d, const float4 e, const float4 f,
                                              const float4 h, float sharp) {
  const float mn4R = fminf(fminf(b.x, fminf(d.x, f.x)), h.x), mx4R = fmaxf(fmaxf(b.x, fmaxf(d.x, f.x)), h.x);
  const float mn4G = fminf(fminf(b.y, fminf(d.y, f.y)), h.y), mx4G = fmaxf(fmaxf(b.y, fmaxf(d.y, f.y)), h.y);
  const float mn4B = fminf(fminf(b.z, fminf(d.z, f.z)), h.z), mx4B = fmaxf(fmaxf(b.z, fmaxf(d.z, f.z)), h.z);
  // limiters need full-precision reciprocals (:748-755)
  const float hitMinR = mn4R * rcp_mode_rcas<U8>(4.0f * mx4R);
  const float hitMinG = mn4G * rcp_mode_rcas<U8>(4.0f * mx4G);
  const float hitMinB = mn4B * rcp_mode_rcas<U8>(4.0f * mx4B);
  const float hitMaxR = (1.0f - mx4R) * rcp_mode_rcas<U8>(4.0f * mn4R + (-4.0f));
  const float hitMaxG = (1.0f - mx4G) * rcp_mode_rcas<U8>(4.0f * mn4G + (-4.0f));
  const float hitMaxB = (1.0f - mx4B) * rcp_mode_rcas<U8>(4.0f * mn4B + (-4.0f));
  const float lobeR = fmaxf(-hitMinR, hitMaxR), lobeG = fmaxf(-hitMinG, hitMaxG), lobeB = fmaxf(-hitMinB, hitMaxB);
  const float lobe =
      fmaxf((float)(-(0.25 - (1.0 / 16.0))), fminf(fmaxf(lobeR, fmaxf(lobeG, lobeB)), 0.0f)) * sharp;
  const float rcpL = prx_med_rcp(4.0f * lobe + 1.0f);
  return make_float3((lobe * b.x + lobe * d.x + lobe * h.x + lobe * f.x + e.x) * rcpL,
                     (lobe * b.y + lobe * d.y + lobe * h.y + lobe * f.y + e.y) * rcpL,
                     (lobe * b.z + lobe * d.z + lobe * h.z + lobe * f.z + e.z) * rcpL);
}

// fast math: (r,g) ride the FP32x2 pipe, b stays scalar; lobe*(b+d+h+f)+e regrouped
__device__ __forceinline__ float3 rcas_filter_fast(const float4 b, const float4 d, const float4 e, const float4 f,
                                                   const float4 h, float sharp) {
  const float mn4R = fminf(fminf(b.x, fminf(d.x, f.x)), h.x), mx4R = fmaxf(fmaxf(b.x, fmaxf(d.x, f.x)), h.x);
  const float mn4G = fminf(fminf(b.y, fminf(d.y, f.y)), h.y), mx4G = fmaxf(fmaxf(b.y, fmaxf(d.y, f.y)), h.y);
  const float mn4B = fminf(fminf(b.z, fminf(d.z, f.z)), h.z), mx4B = fmaxf(fmaxf(b.z, fmaxf(d.z, f.z)), h.z);
  const f2 mx = make_float2(mx4R, mx4G), mn = make_float2(mn4R, mn4G);
  const f2 dMin = mul2(mx, bc(4.0f)), dMax = fma2(mn, bc(4.0f), bc(-4.0f));
  const f2 hitMin = mul2(mn, make_float2(rcp_mode(dMin.x), rcp_mode(dMin.y)));
  const f2 hitMax = mul2(add2(bc(1.0f), make_float2(-mx4R, -mx4G)), make_float2(rcp_mode(dMax.x), rcp_mode(dMax.y)));
  const float hitMinB = mn4B * rcp_mode(4.0f * mx4B);
  const float hitMaxB = (1.0f - mx4B) * rcp_mode(fmaf(4.0f, mn4B, -4.0f));
  const float lobeR = fmaxf(-hitMin.x, hitMax.x), lobeG = fmaxf(-hitMin.y, hitMax.y), lobeB = fmaxf(-hitMinB, hitMaxB);
  const float lobe =
      fmaxf((float)(-(0.25 - (1.0 / 16.0))), fminf(fmaxf(lobeR, fmaxf(lobeG, lobeB)), 0.0f)) * sharp;
  const float rcpL = prx_med_rcp(fmaf(4.0f, lobe, 1.0f));
  const f2 sRG = add2(add2(make_float2(b.x, b.y), make_float2(d.x, d.y)), add2(make_float2(h.x, h.y), make_float2(f.x, f.y)));
  const float sB = (b.z + d.z) + (h.z + f.z);
  const f2 pRG = mul2(fma2(sRG, bc(lobe), make_float2(e.x, e.y)), bc(rcpL));
  return make_float3(pRG.x, pRG.y, fmaf(lobe, sB, e.z) * rcpL);
}

template <bool U8>
__device__ __forceinline__ float3 rcas_filter_mode(const float4 b, const float4 d, const float4 e, const float4 f,
                                                   const float4 h, float sharp) {
  if constexpr (kStrict) return rcas_filter<U8>(b, d, e, f, h, sharp);
  else return rcas_filter_fast(b, d, e, f, h, sharp);
}

// four adjacent output texels -> memory; one 128-bit store when the format is 4 bytes wide and alignment allows
template <int FOUT>
__device__ __forceinline__ void store_quad(const ImageRW &dst, bool vec, int x, int y, const float4 (&px)[4]) {
  uint8_t *row = dst.ptr + (size_t)y * dst.pitch;
  if constexpr (FOUT == OVRFSR_FORMAT_RGBA8 || FOUT == OVRFSR_FORMAT_RGB10A2) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (FOUT == OVRFSR_FORMAT_RGBA8)
        w[i] = __byte_perm(__byte_perm(to_unorm8(px[i].x), to_unorm8(px[i].y), 0x0040), __byte_perm(to_unorm8(px[i].z), to_unorm8(px[i].w), 0x0040), 0x5410);
      else
        w[i] = to_unorm<1023>(px[i].x) | (to_unorm<1023>(px[i].y) << 10) | (to_unorm<1023>(px[i].z) << 20) | (to_unorm<3>(px[i].w) << 30);
    }
    if (vec && x + 3 < dst.w) {
      *reinterpret_cast<uint4 *>(row + (size_t)x * 4) = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (x + i < dst.w) reinterpret_cast<uint32_t *>(row)[x + i] = w[i];
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (x + i < dst.w) store_texel<FOUT>(row, x + i, px[i].x, px[i].y, px[i].z, px[i].w);
  }
}

// One CTA: 64x32 output pixels; the (66 x 34) source box arrives by TMA (zero fill outside the image is exactly
// Texture2D.Load's behaviour) and is decoded once into a float4 tile.  One warp per 16x16 group; each lane walks a
// column of 8 rows and keeps the b / e / h texels of the cross in registers, so a pixel costs 3 shared loads, not 5.
// One tile per CTA on purpose: at 44 registers and 46 KB four CTAs share an SM and the hardware scheduler balances the
// 2808 tiles; a persistent variant (double-buffered landing zones, a lane owning 4 adjacent pixels for 128-bit
// stores, 72 registers, 3 CTAs per SM) was measured at 46.8 us against this kernel's 39.1 us per C2 eye
// (profiles/r2_rejected_experiments.md).
// skipOutside (ctx path, EASU ran with EasuArgs::direct): outside-radius groups are already final in dst, so CTAs
// without an inside group return at once and outside groups of mixed tiles store nothing.
// PAIRED = skipOutside, OPQ = opaqueSrc as compile-time variants (the plain dispatch keeps its instruction stream).
template <int FIN, int FOUT, bool TMA, bool PAIRED, bool OPQ>
__global__ void __launch_bounds__(kThreads, 2) rcas_kernel(const __grid_constant__ RcasArgs a,
                                                           const __grid_constant__ CUtensorMap srcMap) {
  __shared__ __align__(128) float4 sC[kRcasTH * kRcasTW];
  __shared__ __align__(128) uint32_t sRaw[TMA ? kRcasTH * kRcasRawW : 1];
  __shared__ uint64_t tileBar;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ox0 = blockIdx.x * kTileW, oy0 = blockIdx.y * kTileH;
  const int sx0 = ox0 - 1, sy0 = oy0 - 1;
  // same UNORM layout in and out: outside-radius texels pass through bit for bit
  constexpr bool kRawCopy = FIN == FOUT && (FIN == OVRFSR_FORMAT_RGBA8 || FIN == OVRFSR_FORMAT_RGB10A2);

  if constexpr (PAIRED) {
    // uniform per CTA: nothing of this tile is inside the radius -> nothing to do (and no TMA load is issued)
    bool any = false;
#pragma unroll
    for (int g = 0; g < 8; ++g)
      any = any || group_inside((blockIdx.x * 4u + (g & 3)) * 16u + 8u, (blockIdx.y * 2u + (g >> 2)) * 16u + 8u, a.centre, a.radiusSq);
    if (!any) return;
  }
  if constexpr (TMA) {
    if (tid == 0) {
      mbar_init(&tileBar, 1);
      fence_barrier_init();
      mbar_arrive_expect_tx(&tileBar, (uint32_t)(kRcasTH * kRcasRawW * 4));
      tma_load_2d(sRaw, &srcMap, ox0 + a.boxX, sy0 + a.y0, &tileBar); // x origin 16-byte aligned: boxShift unused texels on the left
    }
  }
  const uint32_t ggx = blockIdx.x * (kTileW / 16) + (warp & 3), ggy = blockIdx.y * (kTileH / 16) + (warp >> 2);
  const bool inside = group_inside(ggx * 16u + 8u, ggy * 16u + 8u, a.centre, a.radiusSq);

  if constexpr (TMA) {
    // a CTA whose 8 groups are all outside the radius and copy raw bytes needs no decoded tile at all
    const bool rawCopy = kRawCopy && a.tintGB == 1.0f;
    const int needTile = __syncthreads_or(inside || !rawCopy); // also orders the barrier init before the polls
    mbar_wait(&tileBar, 0);
    // the 34 x 66 texels as one flat index: 9 passes of the 256 threads, 97 % of the lanes busy (a row loop per warp with
    // a 32-wide column loop inside keeps 58 %: 66 columns take three column steps, 34 rows five row steps)
    // tile-uniform: the tile reaches over an edge of a rectangle that is smaller than the texture
    const bool zeroEdge = a.zeroOutside && (sx0 < 0 || sy0 < 0 || sx0 + kTileW + 2 > a.src.w || sy0 + kRcasTH > a.src.h);
    if (needTile && !zeroEdge) {
#pragma unroll
      for (int q = tid; q < kRcasTH * (kTileW + 2); q += kThreads) {
        const int ty = q / (kTileW + 2), tx = q - ty * (kTileW + 2);
        float4 c = decode_rgba<FIN>(sRaw[ty * kRcasRawW + tx + a.boxShift]);
        if constexpr (OPQ) c.w = 1.0f;
        sC[ty * kRcasTW + tx] = c;
      }
    } else if (needTile) {
      for (int q = tid; q < kRcasTH * (kTileW + 2); q += kThreads) {
        const int ty = q / (kTileW + 2), tx = q - ty * (kTileW + 2);
        const int gy = sy0 + ty, gx = sx0 + tx;
        float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gy >= 0 && gy < a.src.h && gx >= 0 && gx < a.src.w) {
          c = decode_rgba<FIN>(sRaw[ty * kRcasRawW + tx + a.boxShift]);
          if constexpr (OPQ) c.w = 1.0f;
        }
        sC[ty * kRcasTW + tx] = c;
      }
    }
  } else {
    // Texture2D.Load semantics: out of bounds reads 0 (fsr_rcas.hlsl:18)
#pragma unroll 3
    for (int q = tid; q < kRcasTH * (kTileW + 2); q += kThreads) {
      const int ty = q / (kTileW + 2), tx = q - ty * (kTileW + 2);
      const int gy = sy0 + ty, gx = sx0 + tx;
      float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gy >= 0 && gy < a.src.h && gx >= 0 && gx < a.src.w) {
        c = fetch_texel<FIN>(a.src.ptr + (size_t)gy * a.src.pitch, gx);
        if constexpr (OPQ) c.w = 1.0f;
      }
      sC[ty * kRcasTW + tx] = c;
    }
  }
  __syncthreads();

  const int x = (int)ggx * 16 + (lane & 15);
  if (x >= a.dst.w) return;
  const int y0 = (int)ggy * 16 + (lane >> 4) * 8; // this lane's 8 consecutive rows
  const float4 *p = sC + (y0 - sy0) * kRcasTW + (x - sx0);
  if (inside) {
    float4 b = p[-kRcasTW], e = p[0];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int y = y0 + k;
      if (y >= a.dst.h) break;
      const float4 h = p[kRcasTW], d = p[-1], f = p[1];
      const float3 c = rcas_filter_mode<FIN == OVRFSR_FORMAT_RGBA8 || FIN == OVRFSR_FORMAT_BGRA8>(b, d, e, f, h, a.sharp);
      store_opaque<FOUT>(a.dst.ptr + (size_t)y * a.dst.pitch, x, c.x, c.y, c.z);
      b = e; e = h; p += kRcasTW;
    }
  } else if constexpr (!PAIRED) {
    // OutputTexture[p] = mul * InputTexture[p], alpha included (fsr_rcas.hlsl:45-53)
    if constexpr (TMA && kRawCopy) {
      if (a.tintGB == 1.0f) {
        // debug tint off: mul == 1 and decode -> x1 -> encode is the identity on all 256 (1024, 4) codes (exhaustive
        // check in tests/test_host_logic.py), so the texel bits are copied straight from the TMA landing zone
        const uint32_t *q = sRaw + (y0 - sy0) * kRcasRawW + (x - sx0) + a.boxShift;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int y = y0 + k;
          if (y >= a.dst.h) break;
          reinterpret_cast<uint32_t *>(a.dst.ptr + (size_t)y * a.dst.pitch)[x] = q[k * kRcasRawW];
        }
        return;
      }
    }
    for (int k = 0; k < 8; ++k) {
      const int y = y0 + k;
      if (y >= a.dst.h) break;
      const float4 e = p[k * kRcasTW];
      store_texel<FOUT>(a.dst.ptr + (size_t)y * a.dst.pitch, x, 1.0f * e.x, a.tintGB * e.y, a.tintGB * e.z, 1.0f * e.w);
    }
  }
}

// Device self-test behind ovrfsr_selftest_rcp: every reciprocal operand strict RCAS can see with a UNORM8 source,
// fast sequence vs rcp.rn.  out[0] = number of mismatching operands (must be 0), out[1] = operands checked.
__global__ void rcas_rcp_selftest_kernel(uint32_t *out) {
  const int k = threadIdx.x; // 0..255
  const float v = unorm8((float)k);
  const float x1 = 4.0f * v, x2 = __fadd_rn(__fmul_rn(4.0f, v), -4.0f);
  int bad = 0;
  bad += f2u(rcp_rn_unorm8_operand(x1)) != f2u(__frcp_rn(x1));
  bad += f2u(rcp_rn_unorm8_operand(x2)) != f2u(__frcp_rn(x2));
  atomicAdd(&out[0], (uint32_t)bad);
  atomicAdd(&out[1], 2u);
}

} // inline namespace OVRFSR_MODE_NS
} // namespace ovrfsr
