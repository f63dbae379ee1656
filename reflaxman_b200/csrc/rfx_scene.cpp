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

// (sphereMargin and sphereBox, the boxes of the spheres: rfx_sphere_box.h, shared with the device refit)

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
// leaf is tested without indirection.  parents (optional): per leaf and per pair node, 2 * (its parent's pair node) + side, -1 for the
// root (the bottom-up refit of rfx_mesh.cu).
template <typename WriteSlot>
void packBvh(const std::vector<BvhNode> & nodes, const std::vector<BvhPrim> & prims, int slotFloat4, float pad, WriteSlot writeSlot, PackedBvh & out,
             std::vector<int> * leafParent = nullptr, std::vector<int> * pairParent = nullptr)
{
  std::vector<int> ref;
  const size_t nLeaves = bvhRefs(nodes, ref), nInner = nodes.size() - nLeaves;
  if (leafParent)
  {
    leafParent->assign(nLeaves, -1);
    pairParent->assign(nInner, -1);
    for (size_t i = 0; i < nodes.size(); i++)
      if (nodes[i].b >= 0)
        for (int side = 0; side < 2; side++)
        {
          const int c = side ? nodes[i].b : nodes[i].a;
          if (nodes[c].b < 0) (*leafParent)[(~ref[c]) / 4] = 2 * ref[i] + side;
          else (*pairParent)[ref[c]] = 2 * ref[i] + side;
        }
  }
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
// farOrigins (scenes with a plane, see farGrowthSpheres): a sliver or non-finite triangle gets the box (-inf, +inf) instead, which marks it
// as tested after the walk and kept out of the hierarchy; triReach receives the box R is the diagonal of and kappaMax the largest
// kappa of the triangles that keep a finite box (0 when there is none).
double buildTriBoxes(int n, const float * tris, const float reach[6], float * boxes, bool farOrigins = false, double triReach[6] = nullptr,
                     double * kappaMax = nullptr)
{
  std::vector<TriExtent> e((size_t)n);
  double ulo[3] = { reach[0], reach[1], reach[2] }, uhi[3] = { reach[3], reach[4], reach[5] };
  for (int i = 0; i < n; i++)
  {
    const float * t = tris + 12 * (size_t)i;
    triExtent(t, t + 3, e[i]);
    if (e[i].kappa < 0.0) continue;
    for (int k = 0; k < 3; k++) { ulo[k] = std::min(ulo[k], e[i].lo[k]); uhi[k] = std::max(uhi[k], e[i].hi[k]); }
  }
  const double R = boxDiagonal(ulo, uhi);
  double kmax = 0.0;
  for (int i = 0; i < n; i++)
  {
    triBox(e[i], ulo, uhi, R, farOrigins, boxes + 6 * (size_t)i);
    if (triBoxed(e[i])) kmax = std::max(kmax, e[i].kappa);
  }
  if (triReach)
    for (int k = 0; k < 3; k++) { triReach[k] = ulo[k]; triReach[3 + k] = uhi[k]; }
  if (kappaMax) *kappaMax = kmax;
  return R;
}

// ---- origins outside the reach box (scenes with a plane) ------------------------------------------------------------------------
// The margins above hold for every query whose origin lies in the reach box.  A bounce or shadow ray that starts on an unbounded
// plane can start anywhere; from an origin at Euclidean distance delta outside the box they are too small by at most an amount
// linear in delta, so such a query grows every box it tests by grow * delta_1 (delta_1 >= delta: the sum of the per-axis excesses,
// evaluated on the device rounding upwards), and a query from inside the box grows nothing.
//   Spheres (sphereMargin).  Every centre lies in the reach box, so |v| = |origin - centre| <= R + delta, and the noise bound is
//   h(R + delta) with h(x) = min(3e-7 x^2 / r, 7.7e-4 x).  h is quadratic up to x* = 7.7e-4 r / 3e-7, where its slope is
//   6e-7 x* / r = 2 * 7.7e-4, and linear with slope 7.7e-4 beyond: h(R + delta) <= h(R) + 2 * 7.7e-4 * delta for every r.  The
//   margin is twice h, so it needs 4 * 7.7e-4 * delta more; the slab test's own error (2^-22 |origin| along an axis) grows by
//   2^-22 delta < 1e-6 delta.  growS = 4 * 7.7e-4 + 1e-6.
//   Triangles (buildTriBoxes).  With R the diagonal of the triangle reach box (the reach box joined with every E, which holds v0):
//   |p| <= R + delta and |t d| <= R + delta + dev, so dev <= 20u kappa (R + delta) + 4.2u|A| under the same condition 5u kappa <= 1/2,
//   which does not involve R.  The margin keeps its factor 3 when it grows by 64u kappa delta, plus 1e-6 delta for the slab test:
//   growT = 64u kappa_max + 1e-6, kappa_max over the triangles in the hierarchy (at most 2^19: growT <= 2).  Slivers and non-finite
//   triangles have no such bound: in plane scenes they stay out of the hierarchy and every query tests them after the walk.
// The device widens the slab interval of every box by G |1/d_k| per axis (G = grow * delta_1, rounded upwards; the bounds rounded
// outwards), which is the fused slab test of the box grown by G on every side, with the same clamped reciprocals.
// (farGrowthTris, roundUp and roundOutwards: rfx_tri_setup.h, shared with the device refit)
float farGrowthSpheres() { return roundUp(4.0 * 7.7e-4 + 1e-6); }

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

// (lightFrame, lightDisc, lightGridDims, lightCellsOf, lightTouches and lightGridHeader: rfx_light_grid.h, shared with the device builder
// of rfx_light_grid.cu.)  slots[i]: the leaf slot of prims[i] in the sphere hierarchy (ascending), which fixes the shape of rhoSum.
bool buildLightGrid(const Light & L, const std::vector<const HostObj *> & sph, const std::vector<BvhPrim> & prims, const std::vector<int> & slots,
                    const double blo[3], const double bhi[3], LightGridHost & out)
{
  LightFrame f;
  if (!lightFrame(L, blo, bhi, f)) return false;
  // per sphere: disc centre and radius on the plane
  const size_t n = prims.size();
  std::vector<double> pu(n), pv(n), rho(n);
  double ulo = 1e300, uhi = -1e300, vlo = 1e300, vhi = -1e300, rhoSum = 0.0, blockSum = 0.0;
  int block = 0;
  for (size_t i = 0; i < n; i++)
  {
    const HostObj * o = sph[prims[i].index];
    if (!lightDisc(f, o->center, o->radius, prims[i].m, pu[i], pv[i], rho[i])) return false;
    ulo = std::min(ulo, pu[i] - rho[i]); uhi = std::max(uhi, pu[i] + rho[i]);
    vlo = std::min(vlo, pv[i] - rho[i]); vhi = std::max(vhi, pv[i] + rho[i]);
    // lightRhoSum's shape (rfx_light_grid.h): a block's sum joins the total when the slots leave the block (an empty block adds 0)
    if (slots[i] / LIGHT_GRID_SUM_BLOCK != block) { rhoSum += blockSum; blockSum = 0.0; block = slots[i] / LIGHT_GRID_SUM_BLOCK; }
    blockSum += rho[i];
  }
  rhoSum += blockSum;
  LightGridDims d;
  if (!lightGridDims(ulo, uhi, vlo, vhi, rhoSum, n, d)) return false;
  const int nx = d.nx, ny = d.ny;
  std::vector<uint32_t> count((size_t)nx * ny + 1, 0);
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
      lightCellsOf(d, pu[i], pv[i], rho[i], x0, x1, y0, y1);
      for (int y = y0; y <= y1; y++)
        for (int x = x0; x <= x1; x++)
          if (lightTouches(d, pu[i], pv[i], rho[i], x, y))
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
  lightGridHeader(f, d, g);
  g.cellStart = nullptr; g.itemSphere = nullptr; g.itemIndex = nullptr;
  return true;
}

// The grids of every far light over the drop-point box (blo, bhi), concatenated into img.  prims: the sphere hierarchy's, in the order
// its build left them (its slot order), slots their leaf slots.
void fillLightGrids(const std::vector<Light> & lights, const std::vector<const HostObj *> & sph, const std::vector<BvhPrim> & prims,
                    const std::vector<int> & slots, const double blo[3], const double bhi[3], SceneImage & img)
{
  img.grids.assign(lights.size(), LightGrid());
  img.gridCellOff.assign(lights.size(), 0);
  img.gridItemOff.assign(lights.size(), 0);
  img.gridCells.clear(); img.gridSpheres.clear(); img.gridIndex.clear();
  img.lightGridsBuilt = 0;
  for (size_t li = 0; li < lights.size(); li++)
  {
    LightGridHost lg;
    if (!buildLightGrid(lights[li], sph, prims, slots, blo, bhi, lg)) continue;
    img.grids[li] = lg.g;
    img.gridCellOff[li] = img.gridCells.size(); img.gridItemOff[li] = img.gridSpheres.size();
    img.gridCells.insert(img.gridCells.end(), lg.cellStart.begin(), lg.cellStart.end());
    img.gridSpheres.insert(img.gridSpheres.end(), lg.spheres.begin(), lg.spheres.end());
    img.gridIndex.insert(img.gridIndex.end(), lg.index.begin(), lg.index.end());
    img.lightGridsBuilt++;
  }
  if (!img.lightGridsBuilt) img.grids.clear();
}

// the used leaf slots of a packed sphere hierarchy, ascending: the slots of its prims in the order its build left them
std::vector<int> usedSlots(const PackedBvh & bvh)
{
  std::vector<int> slots;
  for (size_t j = 0; j < bvh.prims.size(); j++)
    if (bvh.prims[j] >= 0) slots.push_back((int)j);
  return slots;
}

// The grids of every far light.  B: the box of every drop point — all objects (with planes present no grid is built: a drop point on
// a plane can lie anywhere), padded for the rounding of a drop point.
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
    double b[6] = { blo[0], blo[1], blo[2], bhi[0], bhi[1], bhi[2] };
    padDropBox(b);
    for (int k = 0; k < 3; k++) { blo[k] = b[k]; bhi[k] = b[3 + k]; img.gridBox[k] = b[k]; img.gridBox[3 + k] = b[3 + k]; }
  }
  fillLightGrids(lights, sph, prims, usedSlots(img.sphBvh), blo, bhi, img);
}

} // namespace

void padDropBox(double b[6])
{
  const double ex = b[3] - b[0], ey = b[4] - b[1], ez = b[5] - b[2];
  const double pad = 1e-3 * sqrt(ex * ex + ey * ey + ez * ez) + 1e-5 * (fabs(b[0]) + fabs(b[1]) + fabs(b[2]) + fabs(b[3]) + fabs(b[4]) + fabs(b[5]));
  for (int k = 0; k < 3; k++) { b[k] -= pad; b[3 + k] += pad; }
}

void sphereDropBox(const HostScene & s, const SceneImage & img, double b[6])
{
  for (int k = 0; k < 3; k++) { b[k] = 1e300; b[3 + k] = -1e300; }
  for (int i : img.sphObj)
  {
    const HostObj & o = s.objs[i];
    for (int k = 0; k < 3; k++)
    {
      b[k] = std::min(b[k], (double)o.center[k] - fabs((double)o.radius));
      b[3 + k] = std::max(b[3 + k], (double)o.center[k] + fabs((double)o.radius));
    }
  }
}

void rebuildLightGrids(const HostScene & s, const SceneImage & img, SceneImage & out)
{
  std::vector<const HostObj *> sph(img.sphObj.size());
  for (size_t i = 0; i < sph.size(); i++) sph[i] = &s.objs[img.sphObj[i]];
  std::vector<BvhPrim> prims;
  prims.reserve(sph.size());
  for (int p : img.sphBvh.prims)
    if (p >= 0)
    {
      BvhPrim q;
      memset(&q, 0, sizeof(q));
      q.index = p;
      q.m = sphereMargin(sph[p]->radius, img.sphR);
      prims.push_back(q);
    }
  const double blo[3] = { img.gridBox[0], img.gridBox[1], img.gridBox[2] }, bhi[3] = { img.gridBox[3], img.gridBox[4], img.gridBox[5] };
  fillLightGrids(s.lights, sph, prims, usedSlots(img.sphBvh), blo, bhi, out);
}

void refreshMeshes(HostScene & s)
{
  for (HostMesh & m : s.meshes)
  {
    if (!m.stale) continue;
    for (size_t k = 0; k < m.idx.size() / 3; k++)
    {
      HostObj & o = s.objs[m.first + k];
      for (int j = 0; j < 3; j++) memcpy(o.triVerts + 3 * j, &m.xyz[3 * (size_t)m.idx[3 * k + j]], 12);
      setupTriangle(o.triVerts, o.tri);
    }
    m.stale = false;
  }
}

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
  img.lightGridsBuilt = 0; img.bvhDepth = 0; img.bvhFloat4 = 0; img.triBvhTris = 0; img.bvhSpheres = 0;
  img.triAlways.clear(); img.far = false;
  img.meshes.clear(); img.meshIdx.clear(); img.triSlot.clear(); img.leafParent.clear(); img.pairParent.clear();
  img.sphSlot.clear(); img.sphLeafParent.clear(); img.sphPairParent.clear(); img.sphR = 0.0;
  memset(img.reach, 0, sizeof(img.reach));
  img.spheres.resize(sph.size()); img.sphObj.resize(sph.size()); img.sphRadius.resize(sph.size());
  for (size_t i = 0; i < sph.size(); i++)
  {
    img.spheres[i] = make_float4(sph[i]->center[0], sph[i]->center[1], sph[i]->center[2], sph[i]->sqRadius);
    img.sphObj[i] = (int)(sph[i] - s.objs.data());
    img.sphRadius[i] = sph[i]->radius;
  }
  // the constant-bank form (built at the end) holds the whole scene
  const bool fitsSmall = sph.size() <= (size_t)SMALL_MAX_SPHERES && tri.size() <= (size_t)SMALL_MAX_TRIS && pla.size() <= (size_t)SMALL_MAX_PLANES &&
                         s.lights.size() <= (size_t)SMALL_MAX_LIGHTS && s.tex.size() <= (size_t)SMALL_MAX_TEX;

  // automatic mode: more than 32 spheres; mode 1: any.  The box margins below are sized for ray origins inside a bounded reach box;
  // next to an (unbounded) plane a drop point can lie anywhere, and a query from outside the box grows the boxes it tests by an
  // amount linear in its distance from the box (farGrowthSpheres): the kernels instantiated with FAR.
  const bool wantBvh = s.bvhMode == 1 ? !sph.empty() : s.bvhMode == 2 ? false : sph.size() > 32;
  // the hierarchy over the triangles: the same rule
  const bool wantTriBvh = s.bvhMode == 1 ? !tri.empty() : s.bvhMode == 2 ? false : tri.size() > 32;
  const bool farOrigins = !pla.empty();
  double R = 0.0;
  if (wantBvh || wantTriBvh)
  {
    // The reach box: every possible ray origin — the camera eye and all drop points (on spheres and triangles) — and every centre.
    // Its diagonal R bounds |origin - centre| in the box margins.  (Planes are unbounded: a drop point on a plane can lie outside the
    // box, and the queries from there grow the boxes (farGrowthSpheres); rfx_set_camera re-flattens the scene when the eye leaves the box.)
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
      p.m = sphereBox(p.c, p.r, R, p.lo, p.hi);
    }
    std::vector<BvhNode> nodes;
    int maxDepth = 0;
    buildBvhRec(nodes, prims, 0, (int)prims.size(), 0, maxDepth);
    if (maxDepth <= BLOB_MAX_BVH_DEPTH)   // the traversal stacks hold 24 entries; a median split of 2^20 spheres is 18 deep
    {
      // leaf slots of one (cx, cy, cz, r^2) each, NaN in the unused ones (their discriminant is NaN: never a hit)
      const float qnan = std::numeric_limits<float>::quiet_NaN();
      // blob scenes: the parents for the refit of rfx_update_spheres (rfx_mesh.cu)
      packBvh(nodes, prims, 1, qnan, [&](int i, float4 * w) { w[0] = img.spheres[i]; }, img.sphBvh,
              fitsSmall ? nullptr : &img.sphLeafParent, fitsSmall ? nullptr : &img.sphPairParent);
      if (!fitsSmall)
      {
        img.sphSlot.assign(sph.size(), -1);
        for (size_t j = 0; j < img.sphBvh.prims.size(); j++)
          if (img.sphBvh.prims[j] >= 0) img.sphSlot[img.sphBvh.prims[j]] = (int)j;
      }
      img.sphR = R;
      img.bvhDepth = maxDepth;
      img.bvhFloat4 = (uint32_t)img.sphBvh.nodes.size();
      h.bvhRoot = img.sphBvh.root;
      h.bvhFloat4 = img.bvhFloat4;
      img.bvhSpheres = sph.size();
      if (s.lightGridsOn && pla.empty() && !s.lights.empty()) buildLightGrids(s.lights, sph, tri, prims, img);
    }
  }
  if (wantTriBvh)
  {
    // The hierarchy over the triangles (buildTriBoxes has the boxes and their margins).  In plane scenes the triangles without a
    // finite box are tested one by one after the walk instead (h.triAlways).
    std::vector<float> tv(tri.size() * 12), boxes(tri.size() * 6);
    for (size_t i = 0; i < tri.size(); i++) { memcpy(&tv[12 * i], tri[i]->tri.v0, 12); memcpy(&tv[12 * i + 3], tri[i]->tri.ax, 36); }
    double triReach[6], kappaMax = 0.0;
    buildTriBoxes((int)tri.size(), tv.data(), img.reach, boxes.data(), farOrigins, triReach, &kappaMax);
    std::vector<BvhPrim> prims;
    std::vector<int> always;
    for (size_t i = 0; i < tri.size(); i++)
    {
      if (farOrigins && std::isinf(boxes[6 * i])) { always.push_back((int)i); continue; }
      BvhPrim p;
      memset(&p, 0, sizeof(p));
      p.index = (int)i;
      for (int k = 0; k < 3; k++)
      {
        p.lo[k] = boxes[6 * i + k]; p.hi[k] = boxes[6 * i + 3 + k];
        p.c[k] = 0.5f * p.lo[k] + 0.5f * p.hi[k];
      }
      prims.push_back(p);
    }
    std::vector<BvhNode> nodes;
    int maxDepth = 0;
    if (!prims.empty()) buildBvhRec(nodes, prims, 0, (int)prims.size(), 0, maxDepth);
    if (!prims.empty() && maxDepth <= BLOB_MAX_BVH_DEPTH)   // deeper (not seen from a median split below ~2^22 triangles): the list walk
    {
      // leaf slots of 3 float4 each (the layout of SmallScene::triPk), all zero in the unused ones, which the exact test's gate
      // |rz| > 2^-63 rejects
      const bool meshes = !s.meshes.empty();
      packBvh(nodes, prims, 3, 0.0f, [&](int i, float4 * w) { packTriangle(tri[i]->tri, w); }, img.triBvh,
              meshes ? &img.leafParent : nullptr, meshes ? &img.pairParent : nullptr);
      if (meshes)
      {
        img.triSlot.assign(tri.size(), -1);
        for (size_t j = 0; j < img.triBvh.prims.size(); j++)
          if (img.triBvh.prims[j] >= 0) img.triSlot[img.triBvh.prims[j]] = (int)j;
        memcpy(img.triUnion, triReach, sizeof(img.triUnion));
      }
      h.triRoot = img.triBvh.root;
      img.triBvhTris = tri.size();
      img.triAlways = always;
      h.nTriAlways = (int)always.size();
      roundOutwards(triReach, h.triReach);
      h.growT = farGrowthTris(kappaMax);
    }
  }
  std::vector<char> inMesh(tri.size(), 0);
  if (!s.meshes.empty())
  {
    // where each mesh's triangles sit in the sorted triangle array (a mesh's triangles are consecutive objects)
    std::vector<int> triOf(s.objs.size(), -1);
    for (size_t i = 0; i < tri.size(); i++) triOf[tri[i] - s.objs.data()] = (int)i;
    for (const HostMesh & m : s.meshes)
    {
      SceneImage::MeshImage mi = { triOf[m.first], (uint32_t)(m.idx.size() / 3), img.meshIdx.size() };
      img.meshes.push_back(mi);
      img.meshIdx.insert(img.meshIdx.end(), m.idx.begin(), m.idx.end());
      memset(&inMesh[mi.triBase], 1, mi.nTris);
    }
  }
  if (img.lightGridsBuilt)   // the drop-point box in parts (rfx_update_mesh and rfx_update_spheres check their current union)
  {
    double * b = img.dropTris;
    for (int k = 0; k < 3; k++) { b[k] = 1e300; b[3 + k] = -1e300; }
    for (size_t i = 0; i < tri.size(); i++)
      if (!inMesh[i])
        for (int v = 0; v < 9; v++) { b[v % 3] = std::min(b[v % 3], (double)tri[i]->triVerts[v]); b[3 + v % 3] = std::max(b[3 + v % 3], (double)tri[i]->triVerts[v]); }
    sphereDropBox(s, img, img.dropSpheres);
  }
  if (farOrigins && (img.bvhSpheres || img.triBvhTris))
  {
    img.far = true;
    memcpy(h.sphReach, img.reach, sizeof(h.sphReach));
    h.growS = farGrowthSpheres();
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
  img.smallOk = fitsSmall;
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
  if (!eyeGridDims(cam, fp.W, fp.H, nx, ny)) return false;
  std::vector<int4> spans(spheres.size());
  cells.assign((size_t)nx * ny + 1, 0);
  for (size_t i = 0; i < spheres.size(); i++)
  {
    const int4 sp = eyeCellSpan(primarySphereBounds(cam, spheres[i]), fp.W, fp.H);   // x0, x1, y0, y1
    for (int y = sp.z; y <= sp.w; y++)
      for (int x = sp.x; x <= sp.y; x++) cells[(size_t)y * nx + x]++;
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
    const int4 & sp = spans[i];
    for (int y = sp.z; y <= sp.w; y++)
      for (int x = sp.x; x <= sp.y; x++)
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
  std::vector<int> slots((size_t)n_spheres);
  for (int i = 0; i < n_spheres; i++) slots[i] = i;                // (one leaf slot per sphere, in order)
  LightGridHost lg;
  counts[0] = counts[1] = 0;
  dims[0] = dims[1] = 0;
  if (!buildLightGrid(L, sph, prims, slots, blo, bhi, lg)) return RFX_OK;      // no grid for this light: dims stay 0
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

int rfx_selftest_far_bounds_host(int n_spheres, const float * spheres, int n_tris, const float * tris, const float reach[6],
                                 float * sphere_boxes, float * tri_boxes, float reaches[12], float grow[2])
{
  if (n_spheres < 0 || n_tris < 0 || (n_spheres && (!spheres || !sphere_boxes)) || (n_tris && (!tris || !tri_boxes)) || !reach || !reaches || !grow)
    return RFX_ERR_ARG;
  // as buildSceneImage: R from the float reach box, the triangle boxes under the plane-scene rule
  const double dx = (double)reach[3] - reach[0], dy = (double)reach[4] - reach[1], dz = (double)reach[5] - reach[2];
  const double R = sqrt(dx * dx + dy * dy + dz * dz);
  for (int i = 0; i < n_spheres; i++) sphereBox(spheres + 4 * i, spheres[4 * i + 3], R, sphere_boxes + 6 * i, sphere_boxes + 6 * i + 3);
  double triReach[6], kappaMax = 0.0;
  buildTriBoxes(n_tris, tris, reach, tri_boxes, true, triReach, &kappaMax);
  memcpy(reaches, reach, 6 * sizeof(float));
  roundOutwards(triReach, reaches + 6);
  grow[0] = farGrowthSpheres(); grow[1] = farGrowthTris(kappaMax);
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
