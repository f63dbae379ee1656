// rfx_light_grid.h — the binary64 arithmetic of a far light's shadow-ray candidate grid (LightGrid), shared by the host builder
// (rfx_scene.cpp buildLightGrid: compiled with -ffp-contract=off) and the device builder (rfx_light_grid.cu: --fmad=false), so a grid
// built on the device is byte for byte the one the host builds for the same spheres, box and R.  Every operation is a correctly rounded
// IEEE operation on both sides; the only reduction whose result depends on its order, the sum of the disc radii, has one fixed shape
// (lightRhoSum).  rfx_scene.cpp, above LightGridHost, has the derivation of the bounds.
#pragma once
#include "rfx_sphere_box.h"

namespace rfx
{

constexpr int LIGHT_GRID_MAX_DIM = 257;                                              // nx, ny <= 256 + 1
constexpr int LIGHT_GRID_CELLS = LIGHT_GRID_MAX_DIM * LIGHT_GRID_MAX_DIM + 1;      // cell offsets of the largest grid
// The shape of the sum of the disc radii: sequential over the used leaf slots inside each block of LIGHT_GRID_SUM_BLOCK consecutive
// slots of the sphere hierarchy, then sequential over the block sums in slot order.
constexpr int LIGHT_GRID_SUM_BLOCK = 256;

// What a light's grid needs besides the spheres: the drop-point box B, its centre and diagonal, the direction l to the light, the bound
// sigma of the angle between a shadow ray and l, and the plane axes u, v across l.
struct LightFrame { double blo[3], bhi[3], cb[3], diag, l[3], sigma, u[3], v[3]; };

// false: the light is inside or near the scene (no grid), or its position or radius is not finite
RFX_HD bool lightFrame(const Light & L, const double blo[3], const double bhi[3], LightFrame & f)
{
  for (int k = 0; k < 3; k++) { f.blo[k] = blo[k]; f.bhi[k] = bhi[k]; }
  for (int k = 0; k < 3; k++) f.cb[k] = 0.5 * (blo[k] + bhi[k]);
  const double ext[3] = { bhi[0] - blo[0], bhi[1] - blo[1], bhi[2] - blo[2] };
  f.diag = sqrt(ext[0] * ext[0] + ext[1] * ext[1] + ext[2] * ext[2]);
  double * l = f.l;
  l[0] = (double)L.ox - f.cb[0]; l[1] = (double)L.oy - f.cb[1]; l[2] = (double)L.oz - f.cb[2];
  const double D = sqrt(l[0] * l[0] + l[1] * l[1] + l[2] * l[2]);
  const double rad = fabs((double)L.radius) * (1.0 + 1e-5);
  if (!(D < 1e300) || !(rad < 1e300) || !(f.diag > 0.0)) return false;
  const double lateral = 0.5 * f.diag + rad;
  if (!(D > 8.0 * lateral)) return false;                       // the light is inside or near the scene: its rays are no bundle
  f.sigma = lateral / (D - lateral) * 1.001 + 1e-6;             // + the float evaluation of the ray on the device
  for (int k = 0; k < 3; k++) l[k] /= D;
  // plane axes
  const int minAxis = fabs(l[0]) <= fabs(l[1]) && fabs(l[0]) <= fabs(l[2]) ? 0 : fabs(l[1]) <= fabs(l[2]) ? 1 : 2;
  double e[3] = { 0, 0, 0 }; e[minAxis] = 1.0;
  double * u = f.u;
  u[0] = l[1] * e[2] - l[2] * e[1]; u[1] = l[2] * e[0] - l[0] * e[2]; u[2] = l[0] * e[1] - l[1] * e[0];
  const double ul = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
  for (int k = 0; k < 3; k++) u[k] /= ul;
  f.v[0] = l[1] * u[2] - l[2] * u[1]; f.v[1] = l[2] * u[0] - l[0] * u[2]; f.v[2] = l[0] * u[1] - l[1] * u[0];
  return true;
}

// The disc of sphere (c, r) on the plane: centre (pu, pv) and radius rho; m its margin in the sphere hierarchy (sphereMargin).  false:
// no finite bound on how far back along l a shadow ray can meet it (the light then gets no grid).
RFX_HD bool lightDisc(const LightFrame & f, const float c[3], float radius, float m, double & pu, double & pv, double & rho)
{
  const double C[3] = { (double)c[0], (double)c[1], (double)c[2] };
  const double r = fabs((double)radius), md = (double)m;
  const double infl = r + md + 1.01 * f.sigma * (f.diag + r);
  // distance from C backwards along l to the boundary of B inflated by infl (C is inside B)
  double sMax = 1e300;
  for (int k = 0; k < 3; k++)
  {
    const double dk = -f.l[k];
    if (dk > 1e-300) sMax = dmin(sMax, (f.bhi[k] + infl - C[k]) / dk);
    else if (dk < -1e-300) sMax = dmin(sMax, (f.blo[k] - infl - C[k]) / dk);
  }
  if (!(sMax < 1e300)) return false;
  sMax = dmax(sMax, 0.0);
  rho = (r + md + f.sigma * sMax) * 1.001 + 1e-5 * f.diag + 1e-6 * (fabs(f.cb[0]) + fabs(f.cb[1]) + fabs(f.cb[2]));   // + the float evaluation of the cell coordinates
  pu = f.u[0] * C[0] + f.u[1] * C[1] + f.u[2] * C[2];
  pv = f.v[0] * C[0] + f.v[1] * C[1] + f.v[2] * C[2];
  return true;
}

// The cells over the discs' extent [ulo, uhi] x [vlo, vhi]: square cells no smaller than 1/256 of the extent nor than 3/4 of the mean
// disc radius (rhoSum over n discs).  false: no disc, or an empty extent (no grid).
struct LightGridDims { double ulo, vlo, cell, inv; int nx, ny; };
RFX_HD bool lightGridDims(double ulo, double uhi, double vlo, double vhi, double rhoSum, uint64_t n, LightGridDims & d)
{
  if (n == 0 || !(uhi > ulo) || !(vhi > vlo)) return false;
  d.ulo = ulo; d.vlo = vlo;
  d.cell = dmax(dmax(uhi - ulo, vhi - vlo) / 256.0, 0.75 * rhoSum / (double)n);
  d.nx = (int)dmin(256.0, ceil((uhi - ulo) / d.cell)) + 1;
  d.ny = (int)dmin(256.0, ceil((vhi - vlo) / d.cell)) + 1;
  d.inv = 1.0 / d.cell;
  return true;
}

// the rectangle of cells [x0, x1] x [y0, y1] around a disc (empty when x0 > x1 or y0 > y1)
RFX_HD void lightCellsOf(const LightGridDims & d, double pu, double pv, double rho, int & x0, int & x1, int & y0, int & y1)
{
  x0 = (int)floor((pu - rho - d.ulo) * d.inv); x0 = x0 < 0 ? 0 : x0;
  x1 = (int)floor((pu + rho - d.ulo) * d.inv); x1 = x1 > d.nx - 1 ? d.nx - 1 : x1;
  y0 = (int)floor((pv - rho - d.vlo) * d.inv); y0 = y0 < 0 ? 0 : y0;
  y1 = (int)floor((pv + rho - d.vlo) * d.inv); y1 = y1 > d.ny - 1 ? d.ny - 1 : y1;
}

// whether a disc meets the square of cell (x, y)
RFX_HD bool lightTouches(const LightGridDims & d, double pu, double pv, double rho, int x, int y)
{
  const double cx0 = d.ulo + x * d.cell, cy0 = d.vlo + y * d.cell;
  const double dx = dmax(dmax(cx0 - pu, pu - (cx0 + d.cell)), 0.0), dy = dmax(dmax(cy0 - pv, pv - (cy0 + d.cell)), 0.0);
  return dx * dx + dy * dy <= rho * rho;
}

// the header floats and sizes of a grid (its pointers are left to the caller)
RFX_HD void lightGridHeader(const LightFrame & f, const LightGridDims & d, LightGrid & g)
{
  for (int k = 0; k < 3; k++) { g.u[k] = (float)(f.u[k] * d.inv); g.v[k] = (float)(f.v[k] * d.inv); }
  g.u[3] = (float)(-d.ulo * d.inv); g.v[3] = (float)(-d.vlo * d.inv);
  g.nx = d.nx; g.ny = d.ny;
}

} // namespace rfx
