// rfx_sphere_box.h — the box of a sphere in the sphere hierarchy, shared by the host scene code (rfx_scene.cpp: compiled with
// -ffp-contract=off) and the sphere refit kernel (rfx_mesh.cu: --fmad=false), so a box computed on the device is bit for bit the one
// the host flatten computes for the same sphere and the same R.  (How the margin grows for ray origins outside the reach box:
// rfx_scene.cpp, above farGrowthSpheres.)
#pragma once
#include "rfx_tri_setup.h"

namespace rfx
{

// Box margin of a sphere of radius r when every ray origin and every centre lies in a box of diagonal R.  The hierarchy must never
// cull a sphere the reference's exact test (Sphere.cpp:49-57) would report, and that test is noisy: with v = origin - centre,
// disc = b*b - 4a*c carries an absolute rounding error of at most ~40 * 2^-24 * a|v|^2 (three-term dot products, the square, the
// product), while a ray that misses the sphere by m has disc = 4a(r^2 - m^2).  A "noise hit" therefore needs m^2 - r^2 < 6e-7 |v|^2,
// i.e. m - r < min(3e-7 |v|^2 / r, 7.7e-4 |v|), and |v| <= R.  The margin is twice that bound, plus 1e-6 R for the device's slab test
// (fused arithmetic with clamped reciprocals: a box plane moves by at most 2^-22 |origin| along its axis).
RFX_HD float sphereMargin(float r, double R)
{
  const double noise = dmin(3e-7 * R * R / dmax((double)r, 1e-30), 7.7e-4 * R);
  return (float)(2.0 * noise + 1e-6 * R);
}

// the box of a sphere in the hierarchy: centre -/+ (r + sphereMargin(r, R)); returns the margin
RFX_HD float sphereBox(const float c[3], float r, double R, float lo[3], float hi[3])
{
  const float m = sphereMargin(r, R);
  for (int k = 0; k < 3; k++) { lo[k] = c[k] - r - m; hi[k] = c[k] + r + m; }
  return m;
}

} // namespace rfx
