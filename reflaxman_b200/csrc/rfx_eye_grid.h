// rfx_eye_grid.h — the binary64 arithmetic of the primary-ray screen bounds of a sphere and of the screen grid of a path's first query
// (EyeGrid), shared by the constant-bank kernel's host-side rectangles (rfx_trace_small.cu makePrimaryCull), the host binning
// (rfx_scene.cpp binEyeGrid: both compiled with -ffp-contract=off) and the device builder (rfx_eye_grid.cu: --fmad=false).  The host's
// results are those of the same source text before it moved here.
//
// The device runs the same double expressions.  sqrt, floor and ceil are correctly rounded on both sides and agree exactly; CUDA's double
// atan2, asin and tan are within a couple of ulp of glibc's but are not guaranteed equal to them.  A rectangle edge computed on the device
// can therefore differ from the host's only where its value lies within ~1e-12 pixels of an integer, and a cell span only where that
// integer is a multiple of 32.  Either side's rectangle is conservative on its own: the margins are CULL_PIX_MARGIN = 3 pixels and
// rEff = 1.001 r + 1e-3 |w|, far above that noise, so either grid lists every sphere a first query can hit.
#pragma once
#include "rfx_tri_setup.h"

namespace rfx
{

// A warp of the constant-bank kernel owns a 4x8 pixel tile; per launch the host bounds, for each sphere, the pixels whose primary ray can
// pass its hit test (rfx_trace_small.cu, above makePrimaryCull, has the derivation).  rect = x0, x1, y0, y1 inclusive; x0 > x1: no pixel.
constexpr int CULL_LO = -(1 << 30), CULL_HI = 1 << 30;
constexpr double CULL_PIX_MARGIN = 3.0;            // sub-samples and jitter reach < 2 pixels past the pixel origin (Render.cpp:177-184)

RFX_HD int4 cullFull() { return make_int4(CULL_LO, CULL_HI, CULL_LO, CULL_HI); }
RFX_HD int4 cullNone() { return make_int4(1, 0, 1, 0); }
RFX_HD int cullClamp(double v)
{
  if (!(v == v)) return 0;
  return v <= (double)CULL_LO ? CULL_LO : v >= (double)CULL_HI ? CULL_HI : (int)v;
}

// A sphere: the tangent planes through the eye that contain the camera's y (x) axis bound its projection in x (y).  The test the
// kernel runs is the float discriminant of Sphere.cpp:49-53, whose rounding noise lets a ray pass that misses the sphere by up to
// sqrt(r^2 + 4e-7 |w|^2) - r: the radius is inflated by 1e-3 r + 1e-3 |w|.
RFX_HD int4 cullSphere(const double * c0, const double * c1, const double * c2, const double * eye, double rz, double wHalf, double hHalf, const float4 & s)
{
  const double w[3] = { (double)s.x - eye[0], (double)s.y - eye[1], (double)s.z - eye[2] };
  const double wl = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  const double r = sqrt(s.w > 0.0f ? (double)s.w : 0.0);
  if (!(wl < 1e300) || !(r < 1e300)) return cullFull();
  const double rEff = r * 1.001 + 1e-3 * wl + 1e-30;
  const double wx = c0[0] * w[0] + c0[1] * w[1] + c0[2] * w[2], wy = c1[0] * w[0] + c1[1] * w[1] + c1[2] * w[2], wz = c2[0] * w[0] + c2[1] * w[1] + c2[2] * w[2];
  int out[4];
  for (int ax = 0; ax < 2; ax++)
  {
    const double a = ax ? wy : wx, half = ax ? hHalf : wHalf;
    const double d2 = sqrt(a * a + wz * wz);
    if (d2 <= rEff) { out[2 * ax] = CULL_LO; out[2 * ax + 1] = CULL_HI; continue; }
    const double th = atan2(a, wz), al = asin(rEff / d2), lim = 1.5707963267948966 - 1e-4;
    const double lo = th - al, hi = th + al;
    if (hi <= -lim || lo >= lim) return cullNone();          // behind the eye in this projection
    out[2 * ax] = lo <= -lim ? CULL_LO : cullClamp(floor(rz * tan(lo) + half - CULL_PIX_MARGIN));
    out[2 * ax + 1] = hi >= lim ? CULL_HI : cullClamp(ceil(rz * tan(hi) + half + CULL_PIX_MARGIN));
  }
  return make_int4(out[0], out[1], out[2], out[3]);
}

// the camera of the bounds, in double
struct PrimaryCamera { double c[3][3], eye[3], rz, wHalf, hHalf, W, H; bool ok; };   // ok = false: no bounds (camera not orthonormal): whole image

RFX_HD PrimaryCamera makePrimaryCamera(const FrameParams & fp)
{
  // ray = rx * c0 + ry * c1 + rz * c2 (Render.cpp:154-156): the bounds need an orthonormal camera (Camera.cpp:24-36 builds one)
  PrimaryCamera cam;
  for (int j = 0; j < 3; j++) { cam.eye[j] = (double)fp.eye[j]; for (int i = 0; i < 3; i++) cam.c[j][i] = (double)fp.view[3 * i + j]; }
  cam.rz = (double)fp.rz; cam.wHalf = (double)fp.wHalf; cam.hHalf = (double)fp.hHalf; cam.W = (double)fp.W; cam.H = (double)fp.H;
  cam.ok = fp.rz > 0.0f && fp.rz < 1e30f && fabs(cam.eye[0]) < 1e30 && fabs(cam.eye[1]) < 1e30 && fabs(cam.eye[2]) < 1e30;
  for (int a = 0; a < 3 && cam.ok; a++)
    for (int b = 0; b < 3; b++)
    {
      const double dot = cam.c[a][0] * cam.c[b][0] + cam.c[a][1] * cam.c[b][1] + cam.c[a][2] * cam.c[b][2];
      if (!(fabs(dot - (a == b ? 1.0 : 0.0)) < 1e-4)) cam.ok = false;
    }
  return cam;
}

// x0, x1, y0, y1 inclusive; x0 > x1: no pixel
RFX_HD int4 primarySphereBounds(const PrimaryCamera & cam, const float4 & sphere)
{
  if (!cam.ok) return cullFull();
  return cullSphere(cam.c[0], cam.c[1], cam.c[2], cam.eye, cam.rz, cam.wHalf, cam.hHalf, sphere);
}

// ---- the screen grid of the first query (EyeGrid) -------------------------------------------------------------------------------------
constexpr int EYE_GRID_SHIFT = 5;                  // 32x32-pixel cells: a 4x8 tile of the kernels lies in one cell
constexpr uint64_t EYE_GRID_MAX_CELLS = 1u << 22;

// The grid's size for a camera and image size; false: no grid (camera not orthonormal, an empty image or more than EYE_GRID_MAX_CELLS
// cells), the first queries walk the hierarchy.  O(1): the host decides it for the device builder too.
RFX_HD bool eyeGridDims(const PrimaryCamera & cam, uint32_t W, uint32_t H, int & nx, int & ny)
{
  if (!cam.ok || W == 0 || H == 0) return false;
  nx = (int)((W + 31u) >> EYE_GRID_SHIFT); ny = (int)((H + 31u) >> EYE_GRID_SHIFT);
  return (uint64_t)nx * ny <= EYE_GRID_MAX_CELLS;
}

// the cells [x0, x1] x [y0, y1] a sphere's rectangle r touches in a W x H image (x0 > x1: none)
RFX_HD int4 eyeCellSpan(const int4 & r, uint32_t W, uint32_t H)
{
  int4 sp = make_int4(1, 0, 1, 0);
  if (r.x <= r.y && r.z <= r.w && r.y >= 0 && r.w >= 0 && r.x < (int)W && r.z < (int)H)
  {
    sp.x = (r.x > 0 ? r.x : 0) >> EYE_GRID_SHIFT; sp.y = (r.y < (int)W - 1 ? r.y : (int)W - 1) >> EYE_GRID_SHIFT;
    sp.z = (r.z > 0 ? r.z : 0) >> EYE_GRID_SHIFT; sp.w = (r.w < (int)H - 1 ? r.w : (int)H - 1) >> EYE_GRID_SHIFT;
  }
  return sp;
}

} // namespace rfx
