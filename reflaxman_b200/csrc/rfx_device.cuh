// rfx_device.cuh — device-side building blocks shared by the trace kernels (un-contracted IEEE binary32 throughout;
// see the ARITHMETIC CONTRACT at the top of rfx_kernels.cu).  Reference citations are path:line under
// /root/reference/src/common.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>
#include "rfx_types.h"

namespace rfx
{

#ifndef RFX_TEXEL_LUT
#define RFX_TEXEL_LUT 0
#endif
#define RFX_VSN 1.08420217248550443e-19f   // sqrtf(FLT_MIN) = 2^-63, reference trace_math.h:17
#define RFX_DELTA 0.0001f                  // reference trace_math.h:18

// =====================================================================================================================
// LCG (reference trace_math.h:36-39): g = 214013*g + 2531011 (mod 2^32), draw = (g >> 16) & 0x7FFF
// =====================================================================================================================
__host__ __device__ __forceinline__ uint32_t lcgJump(uint32_t s, uint32_t n)
{
  // f^n for the affine map f(s) = A s + C by binary powering; the period divides 2^32 so n mod 2^32 is exact
  uint32_t A = 214013u, C = 2531011u;
  while (n)
  {
    if (n & 1u) s = A * s + C;
    C = C * (A + 1u);
    A = A * A;
    n >>= 1;
  }
  return s;
}

// Correctly rounded r / D for the three constant divisors of the path, in 3 FP32 instructions instead of the ~17-cycle
// div.rn sequence: q0 = RN(r * RN(1/D)); rem = fma(-q0, D, r) (exact); q = fma(rem, RN(1/D), q0).
// PROVEN by exhaustion over the whole input domain with exact rational arithmetic (tests/test_oracle.py::
// test_constant_division_is_exact): D = 16383.5 and D = 32767 for r in [0, 32767], D = 255 for r in [0, 255].
__device__ __forceinline__ float divExact(float r, float D, float rcpD)
{
  const float q0 = __fmul_rn(r, rcpD);
  const float rem = __fmaf_rn(-q0, D, r);
  return __fmaf_rn(rem, rcpD, q0);
}
#define RFX_RCP_16383_5 6.103701889514923e-05f   // RN(1 / 16383.5)
#define RFX_RCP_32767 3.0518509447574615e-05f    // RN(1 / 32767)
#define RFX_RCP_255 0.003921568859368563f        // RN(1 / 255)

__device__ __forceinline__ float lcgDrawUnit(uint32_t & s)
{
  s = 214013u * s + 2531011u;
  const int r = (int)((s >> 16) & 0x7FFFu);
  // float(fastrand()) / (float(FAST_RAND_MAX) / 2) - 1.f, Vector3.cpp:182-184
  return divExact(float(r), 16383.5f, RFX_RCP_16383_5) - 1.f;
}

// Accept test of one draw-triple WITHOUT producing the direction (K1 only needs the decision): advances s by three draws.
// With r the 15-bit draw, the reference's component is x = r / 16383.5 - 1 = (2r - 32767) / 32767 exactly in the reals, so
// x^2 + y^2 + z^2 <= 1 is S <= 32767^2 for the integer S = sum (2r - 32767)^2 (< 2^32).  The reference decides on the FLOAT
// evaluation, whose result differs from the real value by at most 1.2e-6 near 1 (correctly rounded division: 1.2e-7 on x; each
// square 3e-7; two additions 2.4e-7) = 1 300 in units of S.  Outside a guard band of 8 192 around 32767^2 the integer test
// therefore gives the reference's decision; inside it (3 triples in a million) the float expression is evaluated as the
// reference does.  rfx_selftest_rng compares the two over every triple of the LCG's whole cycle.
__device__ __forceinline__ bool rngAcceptFloat(int a, int b, int c);
__device__ __forceinline__ bool rngAccept(uint32_t & s)
{
  s = 214013u * s + 2531011u; const int a = (int)((s >> 16) & 0x7FFFu);
  s = 214013u * s + 2531011u; const int b = (int)((s >> 16) & 0x7FFFu);
  s = 214013u * s + 2531011u; const int c = (int)((s >> 16) & 0x7FFFu);
  const int da = 2 * a - 32767, db = 2 * b - 32767, dc = 2 * c - 32767;
  const uint32_t S = (uint32_t)(da * da) + (uint32_t)(db * db) + (uint32_t)(dc * dc);
  const uint32_t R2 = 32767u * 32767u, GUARD = 8192u;
  if (S < R2 - GUARD) return true;
  if (S > R2 + GUARD) return false;
  return rngAcceptFloat(a, b, c);
}

// one draw-triple: advances s by three draws; true when the candidate lies inside the unit sphere (Vector3.cpp:185)
__device__ __forceinline__ bool rngTriple(uint32_t & s, float & x, float & y, float & z)
{
  x = lcgDrawUnit(s);
  y = lcgDrawUnit(s);
  z = lcgDrawUnit(s);
  return !((x * x + y * y) + z * z > 1.f);
}

__device__ __forceinline__ bool rngAcceptFloat(int a, int b, int c)   // the reference's own expression, Vector3.cpp:182-185
{
  const float x = divExact(float(a), 16383.5f, RFX_RCP_16383_5) - 1.f, y = divExact(float(b), 16383.5f, RFX_RCP_16383_5) - 1.f,
              z = divExact(float(c), 16383.5f, RFX_RCP_16383_5) - 1.f;
  return !((x * x + y * y) + z * z > 1.f);
}

// =====================================================================================================================
// vector helpers (float3 by value; un-contracted, reference evaluation order)
// =====================================================================================================================
struct V3 { float x, y, z; };
__device__ __forceinline__ V3 mk(float x, float y, float z) { V3 v; v.x = x; v.y = y; v.z = z; return v; }
__device__ __forceinline__ V3 vadd(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ V3 vsub(V3 a, V3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ V3 vscale(V3 a, float f) { return mk(a.x * f, a.y * f, a.z * f); }
__device__ __forceinline__ float vdot(V3 a, V3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }       // Vector3.cpp:124-127
__device__ __forceinline__ float vsqlen(V3 a) { return (a.x * a.x + a.y * a.y) + a.z * a.z; }           // Vector3.cpp:41-44
__device__ __forceinline__ float vlen(V3 a) { return sqrtf(vsqlen(a)); }                                // Vector3.cpp:36-39
__device__ __forceinline__ V3 normalizeVec(V3 a)   // Vector3.cpp:55-64 == trace_math.cpp:3-12: three true divides, guarded
{
  const float l = vlen(a);
  if (l > RFX_VSN) return mk(a.x / l, a.y / l, a.z / l);
  return a;
}
__device__ __forceinline__ V3 reflectVec(V3 v, V3 n)   // trace_math.cpp:14-23: v - (2*n) * ((v.n)/(n.n))
{
  const float dn = vdot(n, n);
  if (dn > RFX_VSN)
  {
    const float s = vdot(v, n) / dn;
    return mk(v.x - (n.x * 2.0f) * s, v.y - (n.y * 2.0f) * s, v.z - (n.z * 2.0f) * s);
  }
  return v;
}
// powf(x, 3.0f) of Scene.cpp:196 for x in [0, 1]: the double-precision cube rounded once to float is the correctly rounded
// x^3 for every float in [0, 1] (no input double-rounds: tests/test_device_math.py checks every binade exhaustively) and equals
// glibc's powf(x, 3.0f) on 99.94 % of inputs (measured against libm).
__device__ __forceinline__ float cubeLikePowf(float x)
{
  const double d = (double)x;
  return (float)((d * d) * d);
}

// powf(x, y) of Scene.cpp:175 (specular lobe: x in (2^-63, 1], y >= 1).  glibc's powf is correctly rounded in all but a
// vanishing fraction of cases, so the target is RN_float(x^y).  Evaluated in binary64 as 2^(y*log2 x) with ~2^-50 relative
// error, rounded once to float: wrong only when x^y lies within 2^-26 relative of a float rounding boundary, about one
// call in 10^7 (tools/pow_check.cu measures it against CUDA's pow(double, double), < 1 ulp of binary64, rounded to float).  It replaces CUDA's
// pow(double, double), whose 1500 instructions of special-case and extended-precision code evicted the kernel's working
// set from the 32 KB instruction cache.  Requires 0 < x < inf; y finite or +-inf (a NaN exponent is not propagated).
static __device__ __noinline__ float powLikePowf(float xf, float yf)
{
  const double x = (double)xf;                      // exact; float denormals are normal doubles
  int hi = __double2hiint(x);
  const int lo = __double2loint(x);
  int e = (hi >> 20) - 1023;
  hi = (hi & 0x000FFFFF) | 0x3FF00000;              // m in [1, 2)
  if (hi >= 0x3FF6A09F) { hi -= 0x00100000; e += 1; }   // m in [sqrt(1/2), sqrt(2))
  const double m = __hiloint2double(hi, lo);
  // s = (m - 1) / (m + 1): reciprocal seed + two Newton steps, then one residual correction of the quotient
  const double f = m - 1.0, g = m + 1.0;
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(g));
  r = fma(r, fma(-g, r, 1.0), r);
  r = fma(r, fma(-g, r, 1.0), r);
  double s = f * r;
  s = fma(r, fma(-g, s, f), s);
  // ln m = 2 atanh(s) = 2s (1 + s^2/3 + s^4/5 + ...), |s| <= 0.1716: 11 terms leave a 6e-19 relative tail
  const double s2 = s * s;
  double p = 1.0 / 23.0;
  p = fma(p, s2, 1.0 / 21.0);
  p = fma(p, s2, 1.0 / 19.0);
  p = fma(p, s2, 1.0 / 17.0);
  p = fma(p, s2, 1.0 / 15.0);
  p = fma(p, s2, 1.0 / 13.0);
  p = fma(p, s2, 1.0 / 11.0);
  p = fma(p, s2, 1.0 / 9.0);
  p = fma(p, s2, 1.0 / 7.0);
  p = fma(p, s2, 1.0 / 5.0);
  p = fma(p, s2, 1.0 / 3.0);
  const double lnm = fma(s * s2, p, s) * 2.0;       // 2s + 2s^3 p
  // log2 x = e + ln m * log2(e): one fma (the product is not rounded before e is added)
  const double L = fma(lnm, 1.4426950408889634074, (double)e);
  // x == 1 gives L == 0 exactly and powf(1, y) is 1 for every y, also y = +inf (0 * inf would be NaN)
  double z = (L == 0.0) ? 0.0 : (double)yf * L;
  if (!(z > -1000.0)) z = -1000.0;                  // x^y underflows binary32 long before (also absorbs -inf)
  if (!(z < 1000.0)) z = 1000.0;
  const double n = rint(z);
  const double t = (z - n) * 0.69314718055994530942;   // |t| <= 0.3466
  double q = 1.0 / 6227020800.0;                    // Taylor of e^t to t^13: 4e-18 relative tail
  q = fma(q, t, 1.0 / 479001600.0);
  q = fma(q, t, 1.0 / 39916800.0);
  q = fma(q, t, 1.0 / 3628800.0);
  q = fma(q, t, 1.0 / 362880.0);
  q = fma(q, t, 1.0 / 40320.0);
  q = fma(q, t, 1.0 / 5040.0);
  q = fma(q, t, 1.0 / 720.0);
  q = fma(q, t, 1.0 / 120.0);
  q = fma(q, t, 1.0 / 24.0);
  q = fma(q, t, 1.0 / 6.0);
  q = fma(q, t, 0.5);
  q = fma(q, t, 1.0);
  q = fma(q, t, 1.0);
  // scale by 2^n in two steps so that neither factor leaves the binary64 normal range (|n| <= 1000)
  const int ni = (int)n;
  const int n1 = ni / 2, n2 = ni - n1;
  q = q * __hiloint2double((n1 + 1023) << 20, 0);
  q = q * __hiloint2double((n2 + 1023) << 20, 0);
  return (float)q;                                  // cvt.rn.f32.f64: one rounding, also into the float denormal range
}

__device__ __forceinline__ float clamp01(float v) { return v < 0.0f ? 0.0f : v > 1.0f ? 1.0f : v; }   // trace_math.h:24


// =====================================================================================================================
// textures (reference Texture.cpp:216-269) and skybox direction mapping (Skybox.cpp:39-106)
// =====================================================================================================================
__device__ __forceinline__ V3 texel(const TexRef & t, const float * __restrict__ lut, uint32_t x, uint32_t y)
{
  const uint32_t c = __ldg(t.px + (x + t.w * y));
  // Color(ARGB): float(byte) / 255.0f (Color.cpp:11-13)
#if RFX_TEXEL_LUT
  return mk(__ldg(lut + ((c >> 16) & 0xFFu)), __ldg(lut + ((c >> 8) & 0xFFu)), __ldg(lut + (c & 0xFFu)));   // host-computed 256-entry table
#else
  // the exact three-instruction constant division (divExact, proven for every byte) instead of three dependent table loads
  return mk(divExact(float((c >> 16) & 0xFFu), 255.0f, RFX_RCP_255), divExact(float((c >> 8) & 0xFFu), 255.0f, RFX_RCP_255),
            divExact(float(c & 0xFFu), 255.0f, RFX_RCP_255));
#endif
}

// non-empty texture, (u, v) already known to lie in [0, 1]: Texture.cpp:246-268
static __device__ __noinline__ V3 texSampleBilinear(const TexRef & t, const float * __restrict__ lut, float u, float v)
{
  const float cu = u > (1.0f - FLT_EPSILON) ? (1.0f - FLT_EPSILON) : u;
  const float cv = v > (1.0f - FLT_EPSILON) ? (1.0f - FLT_EPSILON) : v;
  const float fx = cu * float(t.w);
  const float fy = cv * float(t.h);
  const uint32_t x = (uint32_t)fx, y = (uint32_t)fy;
  if (x < t.w - 1 && y < t.h - 1)
  {
    const V3 c00 = texel(t, lut, x, y), c01 = texel(t, lut, x, y + 1), c10 = texel(t, lut, x + 1, y), c11 = texel(t, lut, x + 1, y + 1);
    const float uf = fx - floorf(fx), vf = fy - floorf(fy);
    const float uo = 1 - uf, vo = 1 - vf;
    // (c00*uo + c10*uf)*vo + (c01*uo + c11*uf)*vf, Texture.cpp:264
    return mk((c00.x * uo + c10.x * uf) * vo + (c01.x * uo + c11.x * uf) * vf,
              (c00.y * uo + c10.y * uf) * vo + (c01.y * uo + c11.y * uf) * vf,
              (c00.z * uo + c10.z * uf) * vo + (c01.z * uo + c11.z * uf) * vf);
  }
  if (x >= t.w || y >= t.h) return mk(0.0f, 0.0f, 0.0f);   // Texture.cpp:223-224 (unreachable after the clamp)
  return texel(t, lut, x, y);
}

// t == nullptr or t->px == nullptr: empty texture -> the reference's grey checker (Texture.cpp:242-243); the checker and
// the range test are inlined at the call sites, the texel path is a shared subroutine
__device__ __forceinline__ V3 texSampleRef(const TexRef * t, const float * __restrict__ lut, float u, float v)
{
  if (u < 0.0f || u > 1.0f || v < 0.0f || v > 1.0f) return mk(0.0f, 0.0f, 0.0f);
  if (!t || !t->px)
  {
    // int(u*50) % 2 ^ int(v*50) % 2 with u*50, v*50 in [0, 50]: the truncated values are non-negative, so % 2 is & 1
    const float g = ((int(u * 50) ^ int(v * 50)) & 1) ? 0.5f : 0.75f;   // Texture.cpp:243
    return mk(g, g, g);
  }
  return texSampleBilinear(*t, lut, u, v);
}

// direction -> (u, v) in the 4x3 cube-cross atlas, Skybox.cpp:39-103.  Every face evaluates centre +- (p / major) * halfTile;
// a - q*h == a + ((-p)/m)*h bit for bit (negation commutes with IEEE division, multiplication and turns + into -), so the
// face only selects operands and the two divisions are issued once instead of once per face.
// rayLen = ray.length(), passed in by callers that already hold it (same operations, same value)
__device__ __forceinline__ void skyDirToUv(V3 ray, float rayLen, float hw, float hh, float & u, float & v)
{
  const float uLeft = 1.0f / 8.0f, vMid = 3.0f / 6.0f, uFront = 3.0f / 8.0f, uRight = 5.0f / 8.0f, uBack = 7.0f / 8.0f;
  const float vTop = 5.0f / 6.0f, vBottom = 1.0f / 6.0f;
  const V3 n = (rayLen > RFX_VSN) ? mk(ray.x / rayLen, ray.y / rayLen, ray.z / rayLen) : ray;   // trace_math.cpp:3-12
  const float x = n.x, y = n.y, z = n.z;
  const float ax = fabsf(x) + RFX_VSN, ay = fabsf(y) + RFX_VSN, az = fabsf(z) + RFX_VSN;
  float pu, pv, major, cu, cv;
  if (az >= ax && az >= ay)
  {
    major = az; pv = y; cv = vMid;
    if (z > 0) { pu = x; cu = uFront; }          // u = uFront + x / az * hw; v = vMid + y / az * hh
    else       { pu = -x; cu = uBack; }          // u = uBack - x / az * hw
  }
  else if (ax >= ay && ax >= az)
  {
    major = ax; pv = y; cv = vMid;
    if (x > 0) { pu = -z; cu = uRight; }         // u = uRight - z / ax * hw; v = vMid + y / ax * hh
    else       { pu = z; cu = uLeft; }           // u = uLeft + z / ax * hw
  }
  else
  {
    major = ay; pu = x; cu = uFront;             // uTop == uFront == uBottom == 3/8: u = uFront + x / ay * hw
    if (y > 0) { pv = -z; cv = vTop; }           // v = vTop - z / ay * hh
    else       { pv = z; cv = vBottom; }         // v = vBottom + z / ay * hh
  }
  u = cu + pu / major * hw;
  v = cv + pv / major * hh;
}


__device__ __forceinline__ uint32_t packArgb(float r, float g, float b)   // Color::argb, Color.cpp:114-117
{
  return (((uint32_t)(unsigned char)(r * 255.999f)) << 16) | (((uint32_t)(unsigned char)(g * 255.999f)) << 8) |
         ((uint32_t)(unsigned char)(b * 255.999f));
}

#define RFX_SIG(h, ev) ((h) = ((h) ^ (uint32_t)(ev)) * 16777619u)

// =====================================================================================================================
// the pixel loop of Render::renderNext (Render.cpp:136-215), shared by the K2 kernels of both scene families
// =====================================================================================================================
// primary ray through the point (px, py) of the image plane, relative to the image centre (Render.cpp:184-186)
__device__ __forceinline__ V3 primaryRay(const FrameParams & fp, float px, float py)
{
  return mk((px * fp.view[0] + py * fp.view[1]) + fp.rz * fp.view[2],
            (px * fp.view[3] + py * fp.view[4]) + fp.rz * fp.view[5],
            (px * fp.view[6] + py * fp.view[7]) + fp.rz * fp.view[8]);
}

// additive jitter of the pixel with index rel inside the slice: two draws per pixel, Render.cpp:177-178
__device__ __forceinline__ void pixelJitter(const FrameParams & fp, uint32_t rel, float & rndx, float & rndy)
{
  uint32_t s = lcgJump(fp.seedRender, 2u * rel);
  s = 214013u * s + 2531011u; rndx = divExact(float((int)((s >> 16) & 0x7FFFu)), 32767.0f, RFX_RCP_32767);
  s = 214013u * s + 2531011u; rndy = divExact(float((int)((s >> 16) & 0x7FFFu)), 32767.0f, RFX_RCP_32767);
}

// The sn * sn Scene::trace calls of one pixel (Render.cpp:174-196) in the reference's order, ssx outer and ssy inner, so that
// the sum is formed in the same order; then finColor /= float(s*s).  x / 1.0f == x exactly, so sn == 1 skips every divide.
// block: block preview (Render.cpp:158-173: sn == 1, no sub-pixel offset, the colour is the call's own).  Call k uses the random
// state st[k], read through the read-only cache when ldg is set.  trace(ray, randDir, events) is one Scene::trace call.
// Returns the pixel's colour; adds the calls' bounce-loop iterations and shadow rays to bounces and shadow, and raises longest
// to the iterations of the longest call.
template <typename Trace>
__device__ __forceinline__ V3 samplePixel(const FrameParams & fp, float rx, float ry, float rndx, float rndy, int sn, bool block, const uint32_t * st,
                                          bool ldg, uint32_t & bounces, uint32_t & shadow, uint32_t & longest, Trace trace)
{
  V3 fin = mk(0.0f, 0.0f, 0.0f);
  const int nCalls = sn * sn;
  int ssx = 0, ssy = 0;
#pragma unroll 1
  for (int call = 0; call < nCalls; call++)
  {
    uint32_t s = ldg ? __ldg(st + call) : st[call];
    V3 rd;
    rngTriple(s, rd.x, rd.y, rd.z);
    float px = rx, py = ry;
    if (!block)
    {
      // (rx + float(ssx)/s) + rndx, Render.cpp:184
      const float offx = sn == 1 ? 0.0f : float(ssx) / float(sn);
      const float offy = sn == 1 ? 0.0f : float(ssy) / float(sn);
      px = (rx + offx) + rndx;
      py = (ry + offy) + rndy;
    }
    const V3 ray = primaryRay(fp, px, py);
    uint32_t ev = 0;
    const V3 c = trace(ray, rd, ev);
    fin = block ? c : vadd(fin, c);
    bounces += ev & 0xFFFFu; shadow += ev >> 16;
    longest = max(longest, ev & 0xFFFFu);
    if (++ssy == sn) { ssy = 0; ssx++; }
  }
  if (sn != 1)   // Color::operator/=, Color.cpp:50-61 (its guard |s*s| > 2^-63 always holds)
  {
    const float sq = float(nCalls);
    fin = mk(fin.x / sq, fin.y / sq, fin.z / sq);
  }
  return fin;
}

// One-sample framebuffer store of a warp's pixel tile (tileW pixels wide).  The four lanes of a tile row hold four consecutive
// pixels; the first of them stores all four as one 128-bit word when all four are in the image (16-byte aligned when W is a
// multiple of 4 and the frame is), so a warp writes a 4x8 tile with 8 STG.128 and L2 merges them into lines.  out: the lane's
// pixel (any address when !valid).
__device__ __forceinline__ void storeTileRow(uint32_t * out, uint32_t packed, bool valid, uint32_t W, uint32_t tileW)
{
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t p1 = __shfl_down_sync(0xffffffffu, packed, 1), p2 = __shfl_down_sync(0xffffffffu, packed, 2), p3 = __shfl_down_sync(0xffffffffu, packed, 3);
  const uint32_t validMask = __ballot_sync(0xffffffffu, valid);
  const bool rowOfFour = tileW % 4u == 0u && (W & 3u) == 0u && ((validMask >> (lane & ~3u)) & 0xFu) == 0xFu;
  if (rowOfFour)
  {
    if ((lane & 3u) == 0u) *reinterpret_cast<uint4 *>(out) = make_uint4(packed, p1, p2, p3);
  }
  else if (valid) *out = packed;
}

// event counters: one striped atomic pair per warp
__device__ __forceinline__ void flushCounters(unsigned long long * __restrict__ counters, uint32_t nBounces, uint32_t nShadow, uint32_t warpId)
{
  if (!counters) return;   // uniform
  __syncwarp();
  const uint32_t wb = __reduce_add_sync(0xffffffffu, nBounces);
  const uint32_t ws = __reduce_add_sync(0xffffffffu, nShadow);
  if ((threadIdx.x & 31u) == 0u)
  {
    const uint32_t slot = warpId & 31u;
    atomicAdd(&counters[slot * 2], (unsigned long long)wb);
    atomicAdd(&counters[slot * 2 + 1], (unsigned long long)ws);
  }
}

// General K2 body: every mode of Render::renderNext — block preview, grid SSAA, additive jitter, arbitrary pixel slices, float
// image, signatures — one lane per pixel or per block origin.  tiled: the slice is whole rows and each warp renders one tile of
// tileW x (32 / tileW) pixels; threads: the CTA size.  pixelTrace(x, y) returns the Scene::trace call of pixel (x, y),
// trace(ray, randDir, events, sig), where sig is the pixel's hit-path signature.
template <typename PixelTrace>
__device__ __forceinline__ void renderAny(const FrameParams & fp, const uint32_t * __restrict__ sampleStates, float * __restrict__ image,
                                          uint32_t * __restrict__ argbOut, uint32_t * __restrict__ sigOut,
                                          unsigned long long * __restrict__ counters, int tiled, uint32_t tileW, uint32_t threads,
                                          PixelTrace pixelTrace)
{
  uint32_t nBounces = 0, nShadow = 0;
  const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;

  // ---- which pixel does this lane own, and how many Scene::trace calls does it make
  const bool blockMode = fp.sampleNum < 0;                 // block preview, Render.cpp:158-173
  const uint32_t blk = blockMode ? (uint32_t)(-fp.sampleNum) : 1u;
  const int sn = blockMode ? 1 : fp.sampleNum;             // grid SSAA factor, Render.cpp:174-196
  uint32_t x, y;
  bool valid;
  uint64_t firstState;                                     // index of this lane's first ranked random state
  if (blockMode)
  {
    // gid enumerates block origins in scan order starting at rank fp.firstRank
    const uint32_t bw = (fp.W + blk - 1) / blk;
    const uint64_t k = fp.firstRank + gid;
    y = (uint32_t)(k / bw) * blk; x = (uint32_t)(k % bw) * blk;
    valid = y < fp.H && ((uint64_t)y * fp.W + x) < fp.p1;
    firstState = gid;
  }
  else if (tiled)
  {
    // row-aligned slice (a whole frame, a band of rows, or this GPU's strips of a split frame): one pixel tile per warp
    const uint32_t tileH = 32u / tileW;
    const uint32_t tilesX = (fp.W + (tileW - 1u)) / tileW;
    const uint32_t y0 = (uint32_t)(fp.p0 / fp.W), y1 = (uint32_t)(fp.p1 / fp.W);
    const uint32_t warp = (uint32_t)(gid >> 5), lane = threadIdx.x & 31u;
    x = (warp % tilesX) * tileW + (lane % tileW);
    y = y0 + (warp / tilesX) * tileH + (lane / tileW);
    if (fp.stripWorld)
    {
      const uint32_t k = y / fp.stripRows;
      y = (k * fp.stripWorld + fp.stripRank) * fp.stripRows + (y % fp.stripRows);
    }
    valid = x < fp.W && y < y1;
    firstState = (((uint64_t)y * fp.W + x) - fp.p0) * (uint64_t)(sn * sn);
  }
  else
  {
    const uint64_t p = fp.p0 + gid;
    valid = p < fp.p1;
    y = (uint32_t)(p / fp.W); x = (uint32_t)(p % fp.W);
    firstState = gid * (uint64_t)(sn * sn);
  }

  if (valid)
  {
    const uint64_t p = (uint64_t)y * fp.W + x;
    float rndx = 0, rndy = 0;
    if (fp.jitter && !blockMode) pixelJitter(fp, (uint32_t)(p - fp.p0), rndx, rndy);
    uint32_t sig = 2166136261u, longest = 0;
    const auto trace = pixelTrace(x, y);
    const V3 fin = samplePixel(fp, float(x) - fp.wHalf, float(y) - fp.hHalf, rndx, rndy, sn, blockMode, sampleStates + firstState, false,
                               nBounces, nShadow, longest, [&](V3 ray, V3 rd, uint32_t & ev) { return trace(ray, rd, ev, sig); });
    const uint32_t ex = min(x + blk, fp.W), ey = min(y + blk, fp.H);
    const uint32_t packed = packArgb(fin.x, fin.y, fin.z);
#pragma unroll 1
    for (uint32_t qy = y; qy < ey; qy++)
#pragma unroll 1
      for (uint32_t qx = x; qx < ex; qx++)
      {
        const uint64_t q = (uint64_t)qy * fp.W + qx;
        if (image)
        {
          float * px = image + q * 3;
          if (fp.accumulate && !blockMode) { px[0] = px[0] + fin.x; px[1] = px[1] + fin.y; px[2] = px[2] + fin.z; }
          else { px[0] = fin.x; px[1] = fin.y; px[2] = fin.z; }
        }
        if (argbOut) argbOut[q] = packed;
        if (sigOut) sigOut[q] = sig;
      }
  }
  flushCounters(counters, nBounces, nShadow, blockIdx.x * (threads / 32) + (threadIdx.x >> 5));
}

} // namespace rfx
