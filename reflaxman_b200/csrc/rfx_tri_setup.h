// rfx_tri_setup.h — the per-triangle arithmetic shared by the host scene code (rfx_scene.cpp, rfx_capi.cu: compiled with
// -ffp-contract=off) and the mesh-update kernels (rfx_mesh.cu: --fmad=false): the reference's triangle constructor and the box of a
// triangle in the triangle hierarchy.  One definition of each, so a triangle set up or boxed on the device is bit for bit the one the
// host would have made.  Every operation is a correctly rounded IEEE operation on both sides (no contraction, no fast math).
#pragma once
#include "rfx_types.h"

#include <float.h>
#include <math.h>
#include <string.h>
#include <vector_functions.h>

#ifdef __CUDACC__
#define RFX_HD __host__ __device__ inline
#else
#define RFX_HD inline
#endif

namespace rfx
{

constexpr float VSN = 1.08420217248550443e-19f;   // sqrtf(FLT_MIN), reference trace_math.h:17

struct H3 { float x, y, z; };
RFX_HD H3 hsub(H3 a, H3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
RFX_HD H3 hcross(H3 a, H3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }   // Vector3.cpp:136-141
RFX_HD H3 hnormalize(H3 a)   // trace_math.cpp:3-12
{
  const float l = sqrtf((a.x * a.x + a.y * a.y) + a.z * a.z);
  if (l > VSN) return { a.x / l, a.y / l, a.z / l };
  return a;
}

// Matrix33(u, v, n) columns + invert(), reference Matrix33.cpp:10-15, 49-79
RFX_HD void invertColumns(H3 u, H3 v, H3 n, float out[9])
{
  const float _11 = u.x, _12 = v.x, _13 = n.x, _21 = u.y, _22 = v.y, _23 = n.y, _31 = u.z, _32 = v.z, _33 = n.z;
  const float d = (_11 * (_22 * _33 - _32 * _23) + _21 * (_32 * _13 - _12 * _33)) + _31 * (_12 * _23 - _13 * _22);
  if (fabsf(d) > VSN)
  {
    out[0] = (_22 * _33 - _23 * _32) / d; out[1] = (_13 * _32 - _12 * _33) / d; out[2] = (_12 * _23 - _13 * _22) / d;
    out[3] = (_23 * _31 - _21 * _33) / d; out[4] = (_11 * _33 - _13 * _31) / d; out[5] = (_13 * _21 - _11 * _23) / d;
    out[6] = (_21 * _32 - _22 * _31) / d; out[7] = (_12 * _31 - _11 * _32) / d; out[8] = (_11 * _22 - _12 * _21) / d;
  }
  else
    for (int k = 0; k < 9; k++) out[k] = (k % 4 == 0) ? 1.0f : 0.0f;
}

// Triangle::Triangle (Triangle.cpp:11-21) of the vertices v[9]: writes t.v0, t.ax and t.n, nothing else (texture fields stay)
RFX_HD void setupTriangle(const float v[9], Triangle & t)
{
  const H3 v0 = { v[0], v[1], v[2] }, v1 = { v[3], v[4], v[5] }, v2 = { v[6], v[7], v[8] };
  const H3 n = hnormalize(hcross(hsub(v1, v0), hsub(v2, v0)));  // Triangle.cpp:13
  const H3 nn = { -n.x, -n.y, -n.z };
  invertColumns(hsub(v2, v0), hsub(v1, v0), nn, t.ax);          // Triangle.cpp:19-20
  t.v0[0] = v0.x; t.v0[1] = v0.y; t.v0[2] = v0.z;
  t.n[0] = n.x; t.n[1] = n.y; t.n[2] = n.z;
}

// a triangle as 3 float4 for the intersection loops (SmallScene::triPk, the leaf slots of the triangle hierarchy)
RFX_HD void packTriangle(const Triangle & t, float4 w[3])
{
  w[0] = make_float4(t.v0[0], t.v0[1], t.v0[2], t.ax[6]);
  w[1] = make_float4(t.ax[7], t.ax[8], t.ax[0], t.ax[1]);
  w[2] = make_float4(t.ax[2], t.ax[3], t.ax[4], t.ax[5]);
}

// std::min / std::max, NaN handling included, in both compilations
RFX_HD double dmin(double a, double b) { return (b < a) ? b : a; }
RFX_HD double dmax(double a, double b) { return (a < b) ? b : a; }
RFX_HD float roundDown(double v) { float f = (float)v; if ((double)f > v) f = nextafterf(f, -FLT_MAX); return f; }
RFX_HD float roundUp(double v) { float f = (float)v; if ((double)f < v) f = nextafterf(f, FLT_MAX); return f; }

// A box (lo xyz, hi xyz) rounded outwards to float
RFX_HD void roundOutwards(const double in[6], float out[6])
{
  for (int k = 0; k < 3; k++) { out[k] = roundDown(in[k]); out[3 + k] = roundUp(in[3 + k]); }
}

// growth of the triangle boxes per unit of distance outside the reach box (rfx_scene.cpp, above farGrowthSpheres)
RFX_HD float farGrowthTris(double kappaMax) { return roundUp(64.0 / 16777216.0 * kappaMax + 1e-6); }

// The first half of a triangle's box in the hierarchy (rfx_scene.cpp buildTriBoxes has the derivation): from v0 and axTrans, the box
// of the effective triangle E (lo xyz, hi xyz), |A| and kappa in binary64.  kappa < 0: M or A or E is not finite (no finite E).
struct TriExtent { double lo[3], hi[3], normA, kappa; };
RFX_HD void triExtent(const float v0[3], const float ax[9], TriExtent & r)
{
  double M[9], A[9];
  bool ok = true;
  for (int k = 0; k < 9; k++) { M[k] = ax[k]; ok = ok && isfinite(M[k]); }
  for (int k = 0; k < 3; k++) ok = ok && isfinite((double)v0[k]);
  double det = 0;
  if (ok)
  {
    A[0] = M[4] * M[8] - M[5] * M[7]; A[1] = M[2] * M[7] - M[1] * M[8]; A[2] = M[1] * M[5] - M[2] * M[4];
    A[3] = M[5] * M[6] - M[3] * M[8]; A[4] = M[0] * M[8] - M[2] * M[6]; A[5] = M[2] * M[3] - M[0] * M[5];
    A[6] = M[3] * M[7] - M[4] * M[6]; A[7] = M[1] * M[6] - M[0] * M[7]; A[8] = M[0] * M[4] - M[1] * M[3];
    det = M[0] * A[0] + M[1] * A[3] + M[2] * A[6];
    ok = isfinite(det) && det != 0.0;
  }
  r.kappa = -1.0;
  if (!ok) return;
  double na = 0, kappa = 0;
  for (int k = 0; k < 9; k++) { A[k] /= det; na += A[k] * A[k]; }
  na = sqrt(na);
  for (int k = 0; k < 3; k++)   // |column k of A| * |row k of M|
    kappa += sqrt(A[k] * A[k] + A[3 + k] * A[3 + k] + A[6 + k] * A[6 + k]) * sqrt(M[3 * k] * M[3 * k] + M[3 * k + 1] * M[3 * k + 1] + M[3 * k + 2] * M[3 * k + 2]);
  bool fin = isfinite(na) && isfinite(kappa);
  for (int k = 0; k < 3; k++)
  {
    const double p0 = v0[k], pa = p0 + A[3 * k], pb = p0 + A[3 * k + 1];   // v0, v0 + a, v0 + b (a, b: columns 0 and 1 of A)
    r.lo[k] = dmin(p0, dmin(pa, pb)); r.hi[k] = dmax(p0, dmax(pa, pb));
    fin = fin && isfinite(r.lo[k]) && isfinite(r.hi[k]);
  }
  if (!fin) return;
  r.normA = na; r.kappa = kappa;
}

// Whether a triangle keeps a box of its own (a finite E and no sliver: 16u kappa <= 1/2); its kappa then counts for growT
RFX_HD bool triBoxed(const TriExtent & e) { return e.kappa >= 0.0 && 16.0 / 16777216.0 * e.kappa <= 0.5; }

// The second half: the box, E's inflated by 64u (kappa R + |A|) + 1e-6 R and rounded outwards, R the diagonal of the union box
// (ulo, uhi) of the reach box and every E.  A triangle that is not triBoxed gets the union box, or (-inf, +inf) in scenes with a plane
// (farOrigins: tested after the walk instead).
RFX_HD void triBox(const TriExtent & e, const double ulo[3], const double uhi[3], double R, bool farOrigins, float b[6])
{
  if (!triBoxed(e))
  {
    for (int k = 0; k < 3; k++)
      if (farOrigins) { b[k] = -INFINITY; b[3 + k] = INFINITY; }
      else { b[k] = roundDown(ulo[k]); b[3 + k] = roundUp(uhi[k]); }
    return;
  }
  const double m = 64.0 / 16777216.0 * (e.kappa * R + e.normA) + 1e-6 * R;
  for (int k = 0; k < 3; k++) { b[k] = roundDown(e.lo[k] - m); b[3 + k] = roundUp(e.hi[k] + m); }
}

// the diagonal of a box (lo xyz, hi xyz)
RFX_HD double boxDiagonal(const double lo[3], const double hi[3])
{
  const double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
  return sqrt(dx * dx + dy * dy + dz * dz);
}

// An order-preserving integer encoding of a double (not NaN): atomicMin / atomicMax on the codes are min / max on the values
RFX_HD unsigned long long orderedCode(double v)
{
  unsigned long long b;
  memcpy(&b, &v, 8);
  return (b >> 63) ? ~b : b | 0x8000000000000000ull;
}
RFX_HD double orderedValue(unsigned long long c)
{
  const unsigned long long b = (c >> 63) ? c & 0x7FFFFFFFFFFFFFFFull : ~c;
  double v;
  memcpy(&v, &b, 8);
  return v;
}

} // namespace rfx
