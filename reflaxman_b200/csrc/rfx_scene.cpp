// rfx_scene.cpp — host-side scene flattening (rfx_scene.h) and the pure host self-tests of its bounds.  No CUDA runtime call.
#include "../../include/reflax_c.h"
#include "rfx_kernels.h"
#include "rfx_scene.h"

#include <vector_functions.h>
#include <string.h>
#include <algorithm>
#include <limits>

namespace rfx
{

void invertColumns(H3 u, H3 v, H3 n, float out[9])
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
  {
    const float id[9] = { 1, 0, 0, 0, 1, 0, 0, 0, 1 };
    memcpy(out, id, sizeof(id));
  }
}

Material makeMaterial(int mtype, const float rgb[3], float refl, float transp, int order)
{
  Material m;
  m.r = rgb[0]; m.g = rgb[1]; m.b = rgb[2];
  m.reflectivity = clampf(refl, 0.0f, 1.0f);
  (void)transp;   // clamped and stored by the reference, never read by the tracer (SURVEY §2 #7)
  m.type = mtype ? 1 : 0;
  m.order = order;
  m.tex = -1;
  m.pad = 0;
  return m;
}

FrameParams frameFromCamera(const float eye[3], const float view[9], float fov, uint32_t W, uint32_t H)
{
  FrameParams fp;
  memset(&fp, 0, sizeof(fp));
  memcpy(fp.eye, eye, sizeof(fp.eye));
  memcpy(fp.view, view, sizeof(fp.view));
  fp.rz = float(W) / 2.0f / tanf(fov / 2.0f);            // Render.cpp:148-150
  fp.wHalf = W / 2.0f;
  fp.hHalf = H / 2.0f;
  fp.W = W; fp.H = H;
  return fp;
}

namespace
{

template <typename T> inline size_t align16(T v) { return ((size_t)v + 15) & ~(size_t)15; }

// a triangle as 3 float4 for the intersection loops (SmallScene::triPk, the leaf slots of the triangle hierarchy)
void packTriangle(const Triangle & t, float4 w[3])
{
  w[0] = make_float4(t.v0[0], t.v0[1], t.v0[2], t.ax[6]);
  w[1] = make_float4(t.ax[7], t.ax[8], t.ax[0], t.ax[1]);
  w[2] = make_float4(t.ax[2], t.ax[3], t.ax[4], t.ax[5]);
}

// ---- bounding-volume hierarchies over the spheres and over the triangles of big scenes (SURVEY f-3) ---------------------------
// Median split on the widest centroid axis, leaves of <= 4 primitives, each primitive's box inflated by its margin.  A hierarchy
// only selects which primitives receive the exact reference test on the device; it never decides a hit.
struct BvhNode { float lo[3], hi[3]; int a, b; };
struct BvhPrim
{
  float c[3], r, m;         // spheres: centre (the split key), radius, box margin (sphereMargin); triangles: c = centre of the box
  int index;                // position in the sorted sphere / triangle array (the split's tie-break)
  float lo[3], hi[3];       // the box: spheres c -/+ r -/+ m, triangles buildTriBoxes
};

// Box margin of a sphere of radius r when every ray origin and every centre lies in a box of diagonal R.  The hierarchy must never
// cull a sphere the reference's exact test (Sphere.cpp:49-57) would report, and that test is noisy: with v = origin - centre,
// disc = b*b - 4a*c carries an absolute rounding error of at most ~40 * 2^-24 * a|v|^2 (three-term dot products, the square, the
// product), while a ray that misses the sphere by m has disc = 4a(r^2 - m^2).  A "noise hit" therefore needs m^2 - r^2 < 6e-7 |v|^2,
// i.e. m - r < min(3e-7 |v|^2 / r, 7.7e-4 |v|), and |v| <= R.  The margin is twice that bound, plus 1e-6 R for the device's slab test
// (fused arithmetic with clamped reciprocals: a box plane moves by at most 2^-22 |origin| along its axis).
float sphereMargin(float r, double R)
{
  const double noise = std::min(3e-7 * R * R / std::max((double)r, 1e-30), 7.7e-4 * R);
  return (float)(2.0 * noise + 1e-6 * R);
}

int buildBvhRec(std::vector<BvhNode> & nodes, std::vector<BvhPrim> & prims, int begin, int end, int depth, int & maxDepth)
{
  const int me = (int)nodes.size();
  nodes.push_back(BvhNode());
  maxDepth = std::max(maxDepth, depth);
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX }, clo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, chi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  for (int i = begin; i < end; i++)
    for (int k = 0; k < 3; k++)
    {
      lo[k] = std::min(lo[k], prims[i].lo[k]);
      hi[k] = std::max(hi[k], prims[i].hi[k]);
      clo[k] = std::min(clo[k], prims[i].c[k]);
      chi[k] = std::max(chi[k], prims[i].c[k]);
    }
  BvhNode n;
  memcpy(n.lo, lo, sizeof(lo)); memcpy(n.hi, hi, sizeof(hi));
  if (end - begin <= 4)
  {
    n.a = begin; n.b = -(end - begin);
    nodes[me] = n;
    return me;
  }
  int axis = 0;
  if (chi[1] - clo[1] > chi[axis] - clo[axis]) axis = 1;
  if (chi[2] - clo[2] > chi[axis] - clo[axis]) axis = 2;
  const int mid = (begin + end) / 2;
  std::nth_element(prims.begin() + begin, prims.begin() + mid, prims.begin() + end,
                   [axis](const BvhPrim & x, const BvhPrim & y) { return x.c[axis] < y.c[axis] || (x.c[axis] == y.c[axis] && x.index < y.index); });
  n.a = buildBvhRec(nodes, prims, begin, mid, depth + 1, maxDepth);
  n.b = buildBvhRec(nodes, prims, mid, end, depth + 1, maxDepth);
  nodes[me] = n;
  return me;
}

// Device form of a hierarchy: refs (leaf: ~(first slot), 4 slots per leaf in node order; inner node: its pair-node index) and the
// pair nodes {lo_a.xyz, ref_a} {hi_a.xyz, ref_b} {lo_b.xyz, -} {hi_b.xyz, -}, 4 float4 each, written to pairs
size_t bvhRefs(const std::vector<BvhNode> & nodes, std::vector<int> & ref)
{
  size_t nLeaves = 0;
  for (const BvhNode & n : nodes) nLeaves += n.b < 0;
  ref.resize(nodes.size());
  int inner = 0, lf = 0;
  for (size_t i = 0; i < nodes.size(); i++) ref[i] = nodes[i].b < 0 ? ~(4 * lf++) : inner++;
  return nLeaves;
}

void writePairNode(const std::vector<BvhNode> & nodes, const std::vector<int> & ref, size_t i, float4 * pairs)
{
  const BvhNode & ca = nodes[nodes[i].a], & cb = nodes[nodes[i].b];
  float4 * w = pairs + 4 * (size_t)ref[i];
  w[0] = make_float4(ca.lo[0], ca.lo[1], ca.lo[2], 0.0f); w[1] = make_float4(ca.hi[0], ca.hi[1], ca.hi[2], 0.0f);
  w[2] = make_float4(cb.lo[0], cb.lo[1], cb.lo[2], 0.0f); w[3] = make_float4(cb.hi[0], cb.hi[1], cb.hi[2], 0.0f);
  memcpy(&w[0].w, &ref[nodes[i].a], 4); memcpy(&w[1].w, &ref[nodes[i].b], 4);
}

// [leaf slots | pair nodes] of a hierarchy built by buildBvhRec.  Every leaf is 4 slots of slotFloat4 float4s: writeSlot(position in
// the sorted primitive array, slot) fills a used one, unused ones keep pad — which the device's leaf test never accepts — so a whole
// leaf is tested without indirection.
template <typename WriteSlot>
void packBvh(const std::vector<BvhNode> & nodes, const std::vector<BvhPrim> & prims, int slotFloat4, float pad, WriteSlot writeSlot, PackedBvh & out)
{
  std::vector<int> ref;
  const size_t nLeaves = bvhRefs(nodes, ref), nInner = nodes.size() - nLeaves;
  out.leafFloat4 = nLeaves * 4 * slotFloat4;
  out.nodes.assign(out.leafFloat4 + nInner * 4, make_float4(pad, pad, pad, pad));
  out.prims.assign(nLeaves * 4, -1);
  size_t leaf = 0;
  for (size_t i = 0; i < nodes.size(); i++)
  {
    if (nodes[i].b >= 0)
    {
      writePairNode(nodes, ref, i, &out.nodes[out.leafFloat4]);
      continue;
    }
    for (int k = 0; k < -nodes[i].b; k++)
    {
      const int p = prims[nodes[i].a + k].index;
      writeSlot(p, &out.nodes[(4 * leaf + k) * slotFloat4]);
      out.prims[4 * leaf + k] = p;
    }
    leaf++;
  }
  out.root = ref[0];
}

// Boxes of the triangle hierarchy.  The box of a triangle must hold every point X = o + t d at which the float test of
// Triangle.cpp:56-68 (rfx_trace_blob.cu intersectBlob) can accept it.  That is not the triangle the user gave: the test reads
// M = axTrans = inverse[v2-v0 | v1-v0 | -n] as rounded to float, and a triangle of zero area (n = 0) gets M = identity
// (invertColumns), which accepts a unit right triangle at v0.  So the box starts from the EFFECTIVE triangle
// E = {v0 + u a + v b : u, v >= 0, u + v <= 1} with [a | b | c] = A = M^-1 (binary64), and is inflated by the test's rounding noise.
//
// Margin.  With u = 2^-24, p = o - v0, M_k the rows of M and U, V, W the exact coordinates M (X - v0) of the exact point X = o + t d
// (t the float root the test computed), the test's float ox, rx (row 0), oy, ry (row 1), oz, rz (row 2) carry errors of at most
// 4u|M_k||p| and 3u|M_k||d| (three-term dot products after the subtraction p), so
//   |u_f - U| <= 4u|M_0||p| + 4u|M_0||t d| + u(1 + u)   (one more rounding each for t * rx and the sum; |u_f| <= 1 when accepted)
//   |W|       <= 5u|M_2||p| + 3u|M_2||t d|              (t = fl(-oz / rz) leaves |oz + t rz| <= u|oz| in the float values)
// and likewise for v_f with M_1.  X = v0 + U a + V b + W c therefore lies within
//   dev <= 5u kappa (|p| + |t d|) + 1.01u(|a| + |b|),   kappa = |a||M_0| + |b||M_1| + |c||M_2|   (>= 3: M_k . A_k = 1)
// of the point v0 + u_f a + v_f b, which is in E up to u(|a| + |b|) (u_f + v_f < 1 is a rounded sum).  (kappa is at most sqrt(3) times
// the condition number |M||A|, and much smaller for a small triangle, whose unit normal column c meets a unit row M_2.)  Let R be the
// diagonal of the box that holds every ray origin and every E (the reach box the sphere margins use, joined with the boxes of all E):
// |p| <= R and |t d| = |X - o| <= R + dev, so
//   dev <= 5u kappa (2R + dev) + 2.1u|A|,   i.e. dev <= 20u kappa R + 4.2u|A|   while 5u kappa <= 1/2   (|A|: Frobenius norm).
// The box is E's inflated by m = 64u (kappa R + |A|) (three times the bound: A is formed in binary64, drop points overshoot their
// surface by a rounding) plus 1e-6 R for the device's fused slab test (as for the spheres), rounded outwards to float.  A triangle
// with 16u kappa > 1/2 (a sliver: kappa above 2^19), or whose M or A is not finite, gets the whole box of reach instead: every
// query from inside it then tests that triangle, which is slow but exact.
// tris: n x (v0[3], ax[9]); reach: lo[3], hi[3]; boxes out: n x (lo[3], hi[3]).  Returns R.
double buildTriBoxes(int n, const float * tris, const float reach[6], float * boxes)
{
  const double u = 1.0 / 16777216.0;
  std::vector<double> e((size_t)n * 8);   // per triangle: E's box (lo xyz, hi xyz), |A|, kappa (negative: no finite E)
  double ulo[3] = { reach[0], reach[1], reach[2] }, uhi[3] = { reach[3], reach[4], reach[5] };
  for (int i = 0; i < n; i++)
  {
    const float * t = tris + 12 * (size_t)i;
    double M[9], A[9];
    bool ok = true;
    for (int k = 0; k < 9; k++) { M[k] = t[3 + k]; ok = ok && std::isfinite(M[k]); }
    for (int k = 0; k < 3; k++) ok = ok && std::isfinite((double)t[k]);
    double det = 0;
    if (ok)
    {
      A[0] = M[4] * M[8] - M[5] * M[7]; A[1] = M[2] * M[7] - M[1] * M[8]; A[2] = M[1] * M[5] - M[2] * M[4];
      A[3] = M[5] * M[6] - M[3] * M[8]; A[4] = M[0] * M[8] - M[2] * M[6]; A[5] = M[2] * M[3] - M[0] * M[5];
      A[6] = M[3] * M[7] - M[4] * M[6]; A[7] = M[1] * M[6] - M[0] * M[7]; A[8] = M[0] * M[4] - M[1] * M[3];
      det = M[0] * A[0] + M[1] * A[3] + M[2] * A[6];
      ok = std::isfinite(det) && det != 0.0;
    }
    double * r = &e[8 * (size_t)i];
    r[7] = -1.0;
    if (!ok) continue;
    double na = 0, kappa = 0;
    for (int k = 0; k < 9; k++) { A[k] /= det; na += A[k] * A[k]; }
    na = sqrt(na);
    for (int k = 0; k < 3; k++)   // |column k of A| * |row k of M|
      kappa += sqrt(A[k] * A[k] + A[3 + k] * A[3 + k] + A[6 + k] * A[6 + k]) * sqrt(M[3 * k] * M[3 * k] + M[3 * k + 1] * M[3 * k + 1] + M[3 * k + 2] * M[3 * k + 2]);
    bool fin = std::isfinite(na) && std::isfinite(kappa);
    for (int k = 0; k < 3; k++)
    {
      const double v0 = t[k], pa = v0 + A[3 * k], pb = v0 + A[3 * k + 1];   // v0, v0 + a, v0 + b (a, b: columns 0 and 1 of A)
      r[k] = std::min(v0, std::min(pa, pb)); r[3 + k] = std::max(v0, std::max(pa, pb));
      fin = fin && std::isfinite(r[k]) && std::isfinite(r[3 + k]);
    }
    if (!fin) continue;
    r[6] = na; r[7] = kappa;
    for (int k = 0; k < 3; k++) { ulo[k] = std::min(ulo[k], r[k]); uhi[k] = std::max(uhi[k], r[3 + k]); }
  }
  const double dx = uhi[0] - ulo[0], dy = uhi[1] - ulo[1], dz = uhi[2] - ulo[2];
  const double R = sqrt(dx * dx + dy * dy + dz * dz);
  auto down = [](double v) { float f = (float)v; if ((double)f > v) f = nextafterf(f, -FLT_MAX); return f; };
  auto up = [](double v) { float f = (float)v; if ((double)f < v) f = nextafterf(f, FLT_MAX); return f; };
  for (int i = 0; i < n; i++)
  {
    const double * r = &e[8 * (size_t)i];
    float * b = boxes + 6 * (size_t)i;
    if (!(r[7] >= 0.0) || !(16.0 * u * r[7] <= 0.5))
    {
      for (int k = 0; k < 3; k++) { b[k] = down(ulo[k]); b[3 + k] = up(uhi[k]); }
      continue;
    }
    const double m = 64.0 * u * (r[7] * R + r[6]) + 1e-6 * R;
    for (int k = 0; k < 3; k++) { b[k] = down(r[k] - m); b[3 + k] = up(r[3 + k] + m); }
  }
  return R;
}

// ---- shadow-ray candidate grids (LightGrid) ---------------------------------------------------------------------------------------
// A shadow ray (Scene.cpp:129) runs from a drop point P — a point of some object, so inside the objects' bounding box B — to
// L + radius * randDir, |randDir| <= 1.  For a light far from the scene all those rays are nearly parallel to l = (L - centre(B)) / |..|:
// the sine of their angle to l is at most sigma = (diag(B)/2 + radius) / (|L - centre(B)| - diag(B)/2 - radius).  Project everything
// along l onto a plane.  The exact test (Sphere.cpp:49-57) can only report sphere (C, r) when the ray's line passes within r + m of C
// (m: the rounding-noise bound the hierarchy's box margins use), at a point X = P + s * dir, s > 0; then
//     |proj(C) - proj(P)|  <=  |C - X| + s * sigma  <=  r + m + sigma * s,
// and s is bounded because P must lie in B: C - s*l is within r + m + 1.01 sigma diag(B) of P, so s is at most the distance from C
// backwards along l to the boundary of B inflated by that much.  The grid cell of proj(P) therefore lists every sphere a shadow ray
// from P can hit; the any-hit query tests that list with the reference's exact arithmetic instead of walking the hierarchy, and its
// answer — is the light occluded — is the same.  (Triangles and planes are tested after the list, as before: one by one, or through
// the triangle hierarchy.)
struct LightGridHost
{
  LightGrid g;
  std::vector<uint32_t> cellStart;
  std::vector<float4> spheres;
  std::vector<int> index;
};

bool buildLightGrid(const Light & L, const std::vector<const HostObj *> & sph, const std::vector<BvhPrim> & prims, const double blo[3], const double bhi[3], LightGridHost & out)
{
  const double cb[3] = { 0.5 * (blo[0] + bhi[0]), 0.5 * (blo[1] + bhi[1]), 0.5 * (blo[2] + bhi[2]) };
  const double ext[3] = { bhi[0] - blo[0], bhi[1] - blo[1], bhi[2] - blo[2] };
  const double diag = sqrt(ext[0] * ext[0] + ext[1] * ext[1] + ext[2] * ext[2]);
  double l[3] = { (double)L.ox - cb[0], (double)L.oy - cb[1], (double)L.oz - cb[2] };
  const double D = sqrt(l[0] * l[0] + l[1] * l[1] + l[2] * l[2]);
  const double rad = fabs((double)L.radius) * (1.0 + 1e-5);
  if (!(D < 1e300) || !(rad < 1e300) || !(diag > 0.0)) return false;
  const double lateral = 0.5 * diag + rad;
  if (!(D > 8.0 * lateral)) return false;                       // the light is inside or near the scene: its rays are no bundle
  const double sigma = lateral / (D - lateral) * 1.001 + 1e-6;   // + the float evaluation of the ray on the device
  for (int k = 0; k < 3; k++) l[k] /= D;
  // plane axes
  const int minAxis = fabs(l[0]) <= fabs(l[1]) && fabs(l[0]) <= fabs(l[2]) ? 0 : fabs(l[1]) <= fabs(l[2]) ? 1 : 2;
  double e[3] = { 0, 0, 0 }; e[minAxis] = 1.0;
  double u[3] = { l[1] * e[2] - l[2] * e[1], l[2] * e[0] - l[0] * e[2], l[0] * e[1] - l[1] * e[0] };
  const double ul = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
  for (int k = 0; k < 3; k++) u[k] /= ul;
  const double v[3] = { l[1] * u[2] - l[2] * u[1], l[2] * u[0] - l[0] * u[2], l[0] * u[1] - l[1] * u[0] };
  // per sphere: disc centre and radius on the plane
  const size_t n = prims.size();
  std::vector<double> pu(n), pv(n), rho(n);
  double ulo = 1e300, uhi = -1e300, vlo = 1e300, vhi = -1e300, rhoSum = 0.0;
  for (size_t i = 0; i < n; i++)
  {
    const HostObj * o = sph[prims[i].index];
    const double C[3] = { (double)o->center[0], (double)o->center[1], (double)o->center[2] };
    const double r = fabs((double)o->radius), m = (double)prims[i].m;
    const double infl = r + m + 1.01 * sigma * (diag + r);
    // distance from C backwards along l to the boundary of B inflated by infl (C is inside B)
    double sMax = 1e300;
    for (int k = 0; k < 3; k++)
    {
      const double dk = -l[k];
      if (dk > 1e-300) sMax = std::min(sMax, (bhi[k] + infl - C[k]) / dk);
      else if (dk < -1e-300) sMax = std::min(sMax, (blo[k] - infl - C[k]) / dk);
    }
    if (!(sMax < 1e300)) return false;
    sMax = std::max(sMax, 0.0);
    rho[i] = (r + m + sigma * sMax) * 1.001 + 1e-5 * diag + 1e-6 * (fabs(cb[0]) + fabs(cb[1]) + fabs(cb[2]));   // + the float evaluation of the cell coordinates
    pu[i] = u[0] * C[0] + u[1] * C[1] + u[2] * C[2];
    pv[i] = v[0] * C[0] + v[1] * C[1] + v[2] * C[2];
    ulo = std::min(ulo, pu[i] - rho[i]); uhi = std::max(uhi, pu[i] + rho[i]);
    vlo = std::min(vlo, pv[i] - rho[i]); vhi = std::max(vhi, pv[i] + rho[i]);
    rhoSum += rho[i];
  }
  if (n == 0 || !(uhi > ulo) || !(vhi > vlo)) return false;
  const double cell = std::max(std::max(uhi - ulo, vhi - vlo) / 256.0, 0.75 * rhoSum / (double)n);
  const int nx = (int)std::min(256.0, ceil((uhi - ulo) / cell)) + 1, ny = (int)std::min(256.0, ceil((vhi - vlo) / cell)) + 1;
  const double inv = 1.0 / cell;
  std::vector<uint32_t> count((size_t)nx * ny + 1, 0);
  auto cellsOf = [&](size_t i, int & x0, int & x1, int & y0, int & y1)
  {
    x0 = std::max(0, (int)floor((pu[i] - rho[i] - ulo) * inv)); x1 = std::min(nx - 1, (int)floor((pu[i] + rho[i] - ulo) * inv));
    y0 = std::max(0, (int)floor((pv[i] - rho[i] - vlo) * inv)); y1 = std::min(ny - 1, (int)floor((pv[i] + rho[i] - vlo) * inv));
  };
  auto touches = [&](size_t i, int x, int y)     // the disc against the cell's square
  {
    const double cx0 = ulo + x * cell, cy0 = vlo + y * cell;
    const double dx = std::max(std::max(cx0 - pu[i], pu[i] - (cx0 + cell)), 0.0), dy = std::max(std::max(cy0 - pv[i], pv[i] - (cy0 + cell)), 0.0);
    return dx * dx + dy * dy <= rho[i] * rho[i];
  };
  for (int pass = 0; pass < 2; pass++)
  {
    if (pass == 1)
    {
      uint32_t run = 0;
      for (size_t c = 0; c < (size_t)nx * ny; c++) { const uint32_t k = count[c]; count[c] = run; run += k; }
      count[(size_t)nx * ny] = run;
      out.cellStart = count;
      out.spheres.resize(run); out.index.resize(run);
    }
    for (size_t i = 0; i < n; i++)
    {
      int x0, x1, y0, y1;
      cellsOf(i, x0, x1, y0, y1);
      for (int y = y0; y <= y1; y++)
        for (int x = x0; x <= x1; x++)
          if (touches(i, x, y))
          {
            const size_t c = (size_t)y * nx + x;
            if (pass == 0) count[c]++;
            else
            {
              const HostObj * o = sph[prims[i].index];
              const uint32_t k = count[c]++;
              out.spheres[k] = make_float4(o->center[0], o->center[1], o->center[2], o->sqRadius);
              out.index[k] = prims[i].index;
            }
          }
    }
  }
  LightGrid & g = out.g;
  for (int k = 0; k < 3; k++) { g.u[k] = (float)(u[k] * inv); g.v[k] = (float)(v[k] * inv); }
  g.u[3] = (float)(-ulo * inv); g.v[3] = (float)(-vlo * inv);
  g.nx = nx; g.ny = ny;
  g.cellStart = nullptr; g.itemSphere = nullptr; g.itemIndex = nullptr;
  return true;
}

// The grids of every far light, concatenated into img.  B: the box of every drop point — all objects (planes are excluded by the
// automatic hierarchy rule; with planes present no grid is built), padded for the rounding of a drop point.  prims: the sphere
// hierarchy's, in the order its build left them.
void buildLightGrids(const std::vector<Light> & lights, const std::vector<const HostObj *> & sph, const std::vector<const HostObj *> & tri,
                     const std::vector<BvhPrim> & prims, SceneImage & img)
{
  double blo[3] = { 1e300, 1e300, 1e300 }, bhi[3] = { -1e300, -1e300, -1e300 };
  for (size_t i = 0; i < sph.size(); i++)
    for (int k = 0; k < 3; k++)
    {
      blo[k] = std::min(blo[k], (double)sph[i]->center[k] - fabs((double)sph[i]->radius));
      bhi[k] = std::max(bhi[k], (double)sph[i]->center[k] + fabs((double)sph[i]->radius));
    }
  for (const HostObj * t : tri)
    for (int v = 0; v < 3; v++)
      for (int k = 0; k < 3; k++)
      {
        blo[k] = std::min(blo[k], (double)t->triVerts[3 * v + k]);
        bhi[k] = std::max(bhi[k], (double)t->triVerts[3 * v + k]);
      }
  {
    const double ex = bhi[0] - blo[0], ey = bhi[1] - blo[1], ez = bhi[2] - blo[2];
    const double pad = 1e-3 * sqrt(ex * ex + ey * ey + ez * ez) + 1e-5 * (fabs(blo[0]) + fabs(blo[1]) + fabs(blo[2]) + fabs(bhi[0]) + fabs(bhi[1]) + fabs(bhi[2]));
    for (int k = 0; k < 3; k++) { blo[k] -= pad; bhi[k] += pad; }
  }
  img.grids.assign(lights.size(), LightGrid());
  img.gridCellOff.assign(lights.size(), 0);
  img.gridItemOff.assign(lights.size(), 0);
  for (size_t li = 0; li < lights.size(); li++)
  {
    LightGridHost lg;
    if (!buildLightGrid(lights[li], sph, prims, blo, bhi, lg)) continue;
    img.grids[li] = lg.g;
    img.gridCellOff[li] = img.gridCells.size(); img.gridItemOff[li] = img.gridSpheres.size();
    img.gridCells.insert(img.gridCells.end(), lg.cellStart.begin(), lg.cellStart.end());
    img.gridSpheres.insert(img.gridSpheres.end(), lg.spheres.begin(), lg.spheres.end());
    img.gridIndex.insert(img.gridIndex.end(), lg.index.begin(), lg.index.end());
    img.lightGridsBuilt++;
  }
  if (!img.lightGridsBuilt) img.grids.clear();
}

} // namespace

int buildSceneImage(const HostScene & s, SceneImage & img, std::string & err)
{
  std::vector<const HostObj *> sph, tri, pla;
  for (const HostObj & o : s.objs) (o.kind == 0 ? sph : o.kind == 1 ? tri : pla).push_back(&o);

  SceneHeader h;
  memset(&h, 0, sizeof(h));   // device pointers stay null
  h.nSpheres = (int)sph.size(); h.nTris = (int)tri.size(); h.nPlanes = (int)pla.size();
  h.nLights = (int)s.lights.size(); h.nTextures = (int)s.tex.size();
  h.skyTex = s.skyTex;
  memcpy(h.ambient, s.ambient, sizeof(h.ambient));
  h.ambientPower = s.ambientPower;
  memcpy(h.env, s.env, sizeof(h.env));
  // Skybox::loadTexture / Skybox::Skybox, Skybox.cpp:6-7,21-37
  if (s.skyTex >= 0)
  {
    h.halfTileW = (1.0f / 8.0f - 1.0f / float(s.tex[s.skyTex].w)) - FLT_EPSILON;
    h.halfTileH = (1.0f / 6.0f - 1.0f / float(s.tex[s.skyTex].h)) - FLT_EPSILON;
  }
  else
  {
    h.halfTileW = 1.0f / 8.0f - FLT_EPSILON;
    h.halfTileH = 1.0f / 6.0f - FLT_EPSILON;
  }
  size_t off = align16(sizeof(SceneHeader));
  h.offLights = (uint32_t)off; off = align16(off + sizeof(Light) * s.lights.size());
  h.offSpheres = (uint32_t)off; off = align16(off + sizeof(float) * 4 * sph.size());
  h.offTris = (uint32_t)off; off = align16(off + sizeof(Triangle) * tri.size());
  h.offPlanes = (uint32_t)off; off = align16(off + sizeof(Plane) * pla.size());
  h.offMats = (uint32_t)off; off = align16(off + sizeof(Material) * s.objs.size());
  h.offTex = (uint32_t)off; off = align16(off + sizeof(TexRef) * s.tex.size());
  // the header addresses the blob with 32-bit offsets (every earlier offset is below off)
  if (off > (size_t)UINT32_MAX)
  {
    err = "scene too large: the blob exceeds 4 GB";
    return RFX_ERR_ARG;
  }
  h.bytes = (uint32_t)off;
  img.sphBvh.nodes.clear(); img.sphBvh.prims.clear(); img.triBvh.nodes.clear(); img.triBvh.prims.clear();
  img.grids.clear(); img.gridCells.clear(); img.gridSpheres.clear(); img.gridIndex.clear();
  img.lightGridsBuilt = 0; img.bvhDepth = 0; img.bvhFloat4 = 0; img.triBvhTris = 0;
  memset(img.reach, 0, sizeof(img.reach));
  img.spheres.resize(sph.size());
  for (size_t i = 0; i < sph.size(); i++) img.spheres[i] = make_float4(sph[i]->center[0], sph[i]->center[1], sph[i]->center[2], sph[i]->sqRadius);

  // automatic mode: more than 32 spheres, and no planes — a drop point on an (unbounded) plane can lie anywhere, so the box margins
  // below, which are sized for ray origins inside a bounded region, could not be guaranteed (the reference's Scene cannot hold
  // planes at all).  Mode 1 builds it for any sphere, but never next to a plane either: a bounce off the plane far outside the
  // reach box would walk boxes whose margins do not cover its origin and could lose an occluder or a hit the list walk finds.
  const bool wantBvh = pla.empty() && (s.bvhMode == 1 ? !sph.empty() : s.bvhMode == 2 ? false : sph.size() > 32);
  // the hierarchy over the triangles: the same automatic rule; mode 1 builds it for any triangle, but never next to a plane (its
  // margins need bounded drop points)
  const bool wantTriBvh = pla.empty() && (s.bvhMode == 1 ? !tri.empty() : s.bvhMode == 2 ? false : tri.size() > 32);
  double R = 0.0;
  if (wantBvh || wantTriBvh)
  {
    // The reach box: every possible ray origin — the camera eye and all drop points (on spheres and triangles) — and every centre.
    // Its diagonal R bounds |origin - centre| in the box margins.  (Planes are unbounded: a drop point on a plane can lie outside the
    // box; the reference's Scene cannot hold planes, and rfx_set_camera re-flattens the scene when the eye leaves the box.)
    float lo[3] = { s.eye[0], s.eye[1], s.eye[2] }, hi[3] = { s.eye[0], s.eye[1], s.eye[2] };
    for (int k = 0; k < 3; k++)
      if (s.extraOrigins[k] <= s.extraOrigins[3 + k])   // origins of explicit ray lists (rfx_trace_rays)
      {
        lo[k] = std::min(lo[k], s.extraOrigins[k]);
        hi[k] = std::max(hi[k], s.extraOrigins[3 + k]);
      }
    for (size_t i = 0; i < sph.size(); i++)
      for (int k = 0; k < 3; k++)
      {
        lo[k] = std::min(lo[k], sph[i]->center[k] - sph[i]->radius);
        hi[k] = std::max(hi[k], sph[i]->center[k] + sph[i]->radius);
      }
    for (const HostObj * t : tri)
    {
      for (int v = 0; v < 3; v++)
        for (int k = 0; k < 3; k++)
        {
          lo[k] = std::min(lo[k], t->triVerts[3 * v + k]);
          hi[k] = std::max(hi[k], t->triVerts[3 * v + k]);
        }
    }
    for (int k = 0; k < 3; k++)   // room for the camera to move before the margins have to be recomputed
    {
      const float pad = 0.1f * (hi[k] - lo[k]);
      lo[k] -= pad; hi[k] += pad;
    }
    const double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
    R = sqrt(dx * dx + dy * dy + dz * dz);
    for (int k = 0; k < 3; k++) { img.reach[k] = lo[k]; img.reach[3 + k] = hi[k]; }
  }
  if (wantBvh)
  {
    std::vector<BvhPrim> prims(sph.size());
    for (size_t i = 0; i < sph.size(); i++)
    {
      BvhPrim & p = prims[i];
      memcpy(p.c, sph[i]->center, sizeof(p.c));
      p.r = sph[i]->radius;
      p.index = (int)i;
      p.m = sphereMargin(p.r, R);
      for (int k = 0; k < 3; k++) { p.lo[k] = p.c[k] - p.r - p.m; p.hi[k] = p.c[k] + p.r + p.m; }
    }
    std::vector<BvhNode> nodes;
    int maxDepth = 0;
    buildBvhRec(nodes, prims, 0, (int)prims.size(), 0, maxDepth);
    if (maxDepth <= BLOB_MAX_BVH_DEPTH)   // the traversal stacks hold 24 entries; a median split of 2^20 spheres is 18 deep
    {
      // leaf slots of one (cx, cy, cz, r^2) each, NaN in the unused ones (their discriminant is NaN: never a hit)
      const float qnan = std::numeric_limits<float>::quiet_NaN();
      packBvh(nodes, prims, 1, qnan, [&](int i, float4 * w) { w[0] = img.spheres[i]; }, img.sphBvh);
      img.bvhDepth = maxDepth;
      img.bvhFloat4 = (uint32_t)img.sphBvh.nodes.size();
      h.bvhRoot = img.sphBvh.root;
      h.bvhFloat4 = img.bvhFloat4;
      if (s.lightGridsOn && pla.empty() && !s.lights.empty()) buildLightGrids(s.lights, sph, tri, prims, img);
    }
  }
  if (wantTriBvh)
  {
    // The hierarchy over the triangles (buildTriBoxes has the boxes and their margins)
    std::vector<float> tv(tri.size() * 12), boxes(tri.size() * 6);
    for (size_t i = 0; i < tri.size(); i++) { memcpy(&tv[12 * i], tri[i]->tri.v0, 12); memcpy(&tv[12 * i + 3], tri[i]->tri.ax, 36); }
    buildTriBoxes((int)tri.size(), tv.data(), img.reach, boxes.data());
    std::vector<BvhPrim> prims(tri.size());
    for (size_t i = 0; i < tri.size(); i++)
    {
      BvhPrim & p = prims[i];
      memset(&p, 0, sizeof(p));
      p.index = (int)i;
      for (int k = 0; k < 3; k++)
      {
        p.lo[k] = boxes[6 * i + k]; p.hi[k] = boxes[6 * i + 3 + k];
        p.c[k] = 0.5f * p.lo[k] + 0.5f * p.hi[k];
      }
    }
    std::vector<BvhNode> nodes;
    int maxDepth = 0;
    buildBvhRec(nodes, prims, 0, (int)prims.size(), 0, maxDepth);
    if (maxDepth <= BLOB_MAX_BVH_DEPTH)   // deeper (not seen from a median split below ~2^22 triangles): the list walk
    {
      // leaf slots of 3 float4 each (the layout of SmallScene::triPk), all zero in the unused ones, which the exact test's gate
      // |rz| > 2^-63 rejects
      packBvh(nodes, prims, 3, 0.0f, [&](int i, float4 * w) { packTriangle(tri[i]->tri, w); }, img.triBvh);
      h.triRoot = img.triBvh.root;
      img.triBvhTris = tri.size();
    }
  }

  img.blob.assign(off, 0);
  unsigned char * blob = img.blob.data();
  memcpy(blob, &h, sizeof(h));
  if (!s.lights.empty()) memcpy(blob + h.offLights, s.lights.data(), sizeof(Light) * s.lights.size());
  if (!sph.empty()) memcpy(blob + h.offSpheres, img.spheres.data(), sizeof(float4) * sph.size());
  Material * mats = reinterpret_cast<Material *>(blob + h.offMats);
  size_t mi = 0;
  for (size_t i = 0; i < sph.size(); i++) mats[mi++] = sph[i]->mat;
  for (size_t i = 0; i < tri.size(); i++)
  {
    reinterpret_cast<Triangle *>(blob + h.offTris)[i] = tri[i]->tri;
    mats[mi++] = tri[i]->mat;
  }
  for (size_t i = 0; i < pla.size(); i++)
  {
    reinterpret_cast<Plane *>(blob + h.offPlanes)[i] = pla[i]->plane;
    mats[mi++] = pla[i]->mat;
  }
  for (size_t i = 0; i < s.tex.size(); i++)
  {
    TexRef r;
    r.px = s.tex[i].dev; r.w = s.tex[i].w; r.h = s.tex[i].h;
    reinterpret_cast<TexRef *>(blob + h.offTex)[i] = r;
  }

  // constant-bank form (rfx_trace_small.cu)
  SmallScene & ss = img.small;
  memset(&ss, 0, sizeof(ss));
  img.smallOk = sph.size() <= (size_t)SMALL_MAX_SPHERES && tri.size() <= (size_t)SMALL_MAX_TRIS && pla.size() <= (size_t)SMALL_MAX_PLANES &&
                s.lights.size() <= (size_t)SMALL_MAX_LIGHTS && s.tex.size() <= (size_t)SMALL_MAX_TEX;
  if (!img.smallOk) return RFX_OK;
  ss.nS = h.nSpheres; ss.nT = h.nTris; ss.nP = h.nPlanes; ss.nL = h.nLights;
  ss.skyTex = h.skyTex; ss.halfTileW = h.halfTileW; ss.halfTileH = h.halfTileH;
  ss.ambientPower = h.ambientPower;
  memcpy(ss.ambient, h.ambient, sizeof(ss.ambient));
  memcpy(ss.env, h.env, sizeof(ss.env));
  for (size_t i = 0; i < sph.size(); i++)
  {
    ss.sph[i] = img.spheres[i];
    ss.mat[i] = sph[i]->mat;
  }
  // the sphere loop of the kernels runs over whole quads: pad with NaN records (their discriminant is NaN: never a hit)
  static_assert(SMALL_MAX_SPHERES % 4 == 0, "quads");
  for (size_t i = sph.size(); i % 4 != 0; i++)
  {
    const float qnan = std::numeric_limits<float>::quiet_NaN();
    ss.sph[i] = make_float4(qnan, qnan, qnan, qnan);
    ss.mat[i].order = 0x7FFFFFFF;
    ss.nS = (int)i + 1;
  }
  for (size_t i = 0; i < tri.size(); i++)
  {
    ss.tri[i] = tri[i]->tri; ss.mat[SMALL_MAX_SPHERES + i] = tri[i]->mat;
    packTriangle(tri[i]->tri, ss.triPk[i]);
  }
  for (size_t i = 0; i < pla.size(); i++) { ss.pl[i] = pla[i]->plane; ss.mat[SMALL_MAX_SPHERES + SMALL_MAX_TRIS + i] = pla[i]->mat; }
  for (size_t i = 0; i < s.lights.size(); i++) ss.light[i] = s.lights[i];
  for (size_t i = 0; i < s.tex.size(); i++) { ss.tex[i].px = s.tex[i].dev; ss.tex[i].w = s.tex[i].w; ss.tex[i].h = s.tex[i].h; }
  return RFX_OK;
}

// ---- candidates of the first query of a path (EyeGrid) ------------------------------------------------------------------------------
// Scenes with a sphere hierarchy: every path starts at the eye, so the spheres its first query can hit are the ones whose primary-ray
// screen bounds (primarySphereBounds: the rectangles the constant-bank kernel's tiles use, conservative against the float noise of
// the exact test, SSAA sub-samples and jitter) cover its pixel.  The host bins the rectangles into 32x32-pixel cells per camera; a
// 4x8 tile lies in one cell, so its 32 lanes walk the same short list instead of the hierarchy.  Closest hit over a complete
// candidate list is the hierarchy walk's answer (ties go to the lower insertion index in both).
bool binEyeGrid(const FrameParams & fp, const std::vector<float4> & spheres, int & nx, int & ny, std::vector<uint32_t> & cells,
                std::vector<float4> & items, std::vector<int> & index)
{
  const PrimaryCamera cam = makePrimaryCamera(fp);
  if (!cam.ok || fp.W == 0 || fp.H == 0) return false;
  const int shift = EYE_GRID_SHIFT;
  nx = (int)((fp.W + 31u) >> shift); ny = (int)((fp.H + 31u) >> shift);
  if ((uint64_t)nx * ny > (1u << 22)) return false;
  struct Span { int x0, x1, y0, y1; };
  std::vector<Span> spans(spheres.size());
  cells.assign((size_t)nx * ny + 1, 0);
  for (size_t i = 0; i < spheres.size(); i++)
  {
    const int4 r = primarySphereBounds(cam, spheres[i]);
    Span sp = { 1, 0, 1, 0 };
    if (r.x <= r.y && r.z <= r.w && r.y >= 0 && r.w >= 0 && r.x < (int)fp.W && r.z < (int)fp.H)
    {
      sp.x0 = std::max(r.x, 0) >> shift; sp.x1 = std::min(r.y, (int)fp.W - 1) >> shift;
      sp.y0 = std::max(r.z, 0) >> shift; sp.y1 = std::min(r.w, (int)fp.H - 1) >> shift;
      for (int y = sp.y0; y <= sp.y1; y++)
        for (int x = sp.x0; x <= sp.x1; x++) cells[(size_t)y * nx + x]++;
    }
    spans[i] = sp;
  }
  uint32_t run = 0;
  for (size_t c = 0; c < (size_t)nx * ny; c++) { const uint32_t k = cells[c]; cells[c] = run; run += k; }
  cells[(size_t)nx * ny] = run;
  items.assign(std::max<uint32_t>(run, 1), make_float4(0.0f, 0.0f, 0.0f, 0.0f));
  index.assign(std::max<uint32_t>(run, 1), 0);
  std::vector<uint32_t> fill(cells.begin(), cells.end() - 1);
  for (size_t i = 0; i < spheres.size(); i++)
  {
    const Span & sp = spans[i];
    for (int y = sp.y0; y <= sp.y1; y++)
      for (int x = sp.x0; x <= sp.x1; x++)
      {
        const uint32_t k = fill[(size_t)y * nx + x]++;
        items[k] = spheres[i];
        index[k] = (int)i;
      }
  }
  return true;
}

} // namespace rfx

using namespace rfx;

// =====================================================================================================================
// The host-side bound computations as pure functions (no device, no context), so that the CPU test suite can check them against the
// kernels' float32 expressions evaluated in numpy.
extern "C"
{

int rfx_selftest_primary_bounds_host(const float cam[13], uint32_t width, uint32_t height, int n_spheres, const float * spheres,
                                     int n_tris, const float * tris, int32_t out[96])
{
  if (!cam || !out || n_spheres < 0 || n_spheres > SMALL_MAX_SPHERES || n_tris < 0 || n_tris > SMALL_MAX_TRIS || (n_spheres && !spheres) || (n_tris && !tris) || !width || !height)
    return RFX_ERR_ARG;
  std::vector<SmallScene> holder(1);   // (4 KB: off the stack)
  SmallScene & sc = holder[0];
  memset(&sc, 0, sizeof(sc));
  sc.nS = n_spheres; sc.nT = n_tris;
  for (int i = 0; i < n_spheres; i++) sc.sph[i] = make_float4(spheres[4 * i], spheres[4 * i + 1], spheres[4 * i + 2], spheres[4 * i + 3]);
  for (int k = 0; k < n_tris; k++)
  {
    memcpy(sc.tri[k].v0, tris + 12 * k, 12);
    memcpy(sc.tri[k].ax, tris + 12 * k + 3, 36);
  }
  const PrimaryCull pc = makePrimaryCull(sc, frameFromCamera(cam, cam + 3, cam[12], width, height));
  memcpy(out, pc.rect, sizeof(pc.rect));
  return RFX_OK;
}

int rfx_selftest_light_grid_host(const float light[4], int n_spheres, const float * spheres, const float box[6], float reach_diagonal,
                                 float uv[8], int32_t dims[2], uint32_t * cell_start, uint64_t cell_cap, int32_t * items, uint64_t item_cap,
                                 uint64_t counts[2])
{
  if (!light || !spheres || !box || !uv || !dims || !counts || n_spheres <= 0) return RFX_ERR_ARG;
  std::vector<HostObj> objs((size_t)n_spheres);
  std::vector<const HostObj *> sph((size_t)n_spheres);
  std::vector<BvhPrim> prims((size_t)n_spheres);
  for (int i = 0; i < n_spheres; i++)
  {
    HostObj & o = objs[i];
    memset(&o, 0, sizeof(o));
    memcpy(o.center, spheres + 4 * i, 12);
    o.radius = spheres[4 * i + 3];
    o.sqRadius = o.radius * o.radius;                           // Sphere.cpp:13
    sph[i] = &o;
    BvhPrim & p = prims[i];
    memcpy(p.c, o.center, 12); p.r = o.radius; p.index = i;
    p.m = sphereMargin(p.r, (double)reach_diagonal);
  }
  Light L;
  memset(&L, 0, sizeof(L));
  L.ox = light[0]; L.oy = light[1]; L.oz = light[2]; L.radius = light[3];
  const double blo[3] = { box[0], box[1], box[2] }, bhi[3] = { box[3], box[4], box[5] };
  LightGridHost lg;
  counts[0] = counts[1] = 0;
  dims[0] = dims[1] = 0;
  if (!buildLightGrid(L, sph, prims, blo, bhi, lg)) return RFX_OK;      // no grid for this light: dims stay 0
  memcpy(uv, lg.g.u, 16); memcpy(uv + 4, lg.g.v, 16);
  dims[0] = lg.g.nx; dims[1] = lg.g.ny;
  counts[0] = lg.cellStart.size(); counts[1] = lg.index.size();
  if (cell_start && cell_cap >= lg.cellStart.size()) memcpy(cell_start, lg.cellStart.data(), lg.cellStart.size() * sizeof(uint32_t));
  if (items && item_cap >= lg.index.size() && !lg.index.empty()) memcpy(items, lg.index.data(), lg.index.size() * sizeof(int32_t));
  return RFX_OK;
}

int rfx_selftest_tri_bounds_host(int n, const float * tris, const float reach[6], float * boxes)
{
  if (n < 0 || (n && (!tris || !boxes)) || !reach) return RFX_ERR_ARG;
  buildTriBoxes(n, tris, reach, boxes);
  return RFX_OK;
}

int rfx_selftest_eye_grid_host(const float cam[13], uint32_t width, uint32_t height, int n_spheres, const float * spheres, int32_t dims[3],
                               uint32_t * cell_start, uint64_t cell_cap, int32_t * items, uint64_t item_cap, uint64_t counts[2])
{
  if (!cam || !spheres || !dims || !counts || n_spheres <= 0 || !width || !height) return RFX_ERR_ARG;
  std::vector<float4> sp((size_t)n_spheres);
  for (int i = 0; i < n_spheres; i++) sp[i] = make_float4(spheres[4 * i], spheres[4 * i + 1], spheres[4 * i + 2], spheres[4 * i + 3]);
  int nx = 0, ny = 0;
  std::vector<uint32_t> cells;
  std::vector<float4> rec;
  std::vector<int> index;
  dims[0] = dims[1] = dims[2] = 0; counts[0] = counts[1] = 0;
  if (!binEyeGrid(frameFromCamera(cam, cam + 3, cam[12], width, height), sp, nx, ny, cells, rec, index)) return RFX_OK;   // no grid for this camera: dims stay 0
  dims[0] = nx; dims[1] = ny; dims[2] = EYE_GRID_SHIFT;
  counts[0] = cells.size(); counts[1] = cells.back();
  if (cell_start && cell_cap >= cells.size()) memcpy(cell_start, cells.data(), cells.size() * sizeof(uint32_t));
  if (items && item_cap >= cells.back() && cells.back()) memcpy(items, index.data(), (size_t)cells.back() * sizeof(int32_t));
  return RFX_OK;
}

} // extern "C"
