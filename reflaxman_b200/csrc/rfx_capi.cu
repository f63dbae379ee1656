// rfx_capi.cu — the C ABI of include/reflax_c.h: context, host-side scene flattening, slice scheduling.
//
// Host-side float arithmetic in this file (triangle basis inversion, envColor, skybox half-tile, sqRadius, rz)
// restates what the reference's constructors compute once per object/frame; it is compiled with
// -ffp-contract=off so every operation is the same IEEE binary32 operation the reference's build performs
// (reference Triangle.cpp:11-21,110-120; Matrix33.cpp:10-15,49-79; Scene.cpp:10-15,47-58; Skybox.cpp:21-37;
// Sphere.cpp:9-20; Material.cpp:8-14; OmniLight.cpp:8-14; Render.cpp:148-150).
#include "../../include/reflax_c.h"
#include "rfx_kernels.h"

#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <string.h>
#include <string>
#include <vector>
#include <limits>
#include <algorithm>

using namespace rfx;

namespace
{

const float VSN = 1.08420217248550443e-19f;   // sqrtf(FLT_MIN), reference trace_math.h:17
std::string g_createError;

struct HostTex { uint32_t w = 0, h = 0; std::vector<uint32_t> px; uint32_t * dev = nullptr; bool uploaded = false; };
struct HostObj
{
  int kind;                 // 0 sphere, 1 triangle, 2 plane
  Material mat;             // order = insertion index
  float center[3], sqRadius, radius;
  Triangle tri;
  float triVerts[9];        // the three vertices as given (bounds of the drop points for the BVH margins)
  Plane plane;
};

inline float clampf(float v, float lo, float hi) { return v < lo ? lo : v > hi ? hi : v; }

struct H3 { float x, y, z; };
inline H3 hsub(H3 a, H3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
inline H3 hcross(H3 a, H3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }   // Vector3.cpp:136-141
inline H3 hnormalize(H3 a)   // trace_math.cpp:3-12
{
  const float l = sqrtf((a.x * a.x + a.y * a.y) + a.z * a.z);
  if (l > VSN) return { a.x / l, a.y / l, a.z / l };
  return a;
}

// Matrix33(u, v, n) columns + invert(), reference Matrix33.cpp:10-15, 49-79
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

template <typename T> inline size_t align16(T v) { return ((size_t)v + 15) & ~(size_t)15; }

// ---- bounding-volume hierarchies over the spheres and over the triangles of big scenes (SURVEY f-3) ---------------------------
// Median split on the widest centroid axis, leaves of <= 4 primitives, each primitive's box inflated by its margin.  A hierarchy
// only selects which primitives receive the exact reference test on the device; it never decides a hit.
struct BvhNode { float lo[3], hi[3]; int a, b; };
struct BvhPrim
{
  float c[3], r, m;         // spheres: centre (the split key), radius, box margin (see uploadScene); triangles: c = centre of the box
  int index;                // position in the sorted sphere / triangle array (the split's tie-break)
  float lo[3], hi[3];       // the box: spheres c -/+ r -/+ m, triangles buildTriBoxes
};

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

} // namespace

struct rfx_ctx
{
  int device = 0;
  cudaStream_t stream = nullptr, copyStream[2] = { nullptr, nullptr }, lastStream = nullptr;
  int copyStreams = 1;                      // D2H streams rfx_render_frames alternates between (rfx_set_option "copy_streams")
  cudaDeviceProp prop;
  mutable std::string err;

  // ---- host scene
  float ambient[3] = { 0, 0, 0 }, ambientPower = 0, env[3] = { 0, 0, 0 };
  std::vector<Light> lights;
  std::vector<HostObj> objs;
  std::vector<HostTex> tex;
  int skyTex = -1;
  bool sceneDirty = true;

  // ---- device scene
  unsigned char * dBlob = nullptr; size_t blobCap = 0; uint32_t blobBytes = 0;
  SmallScene small; bool smallOk = false;   // constant-bank form of the same scene, when it fits
  // cost-ordered tile scheduling of the fast kernel (TileOrder, rfx_kernels.h): two list sets, used alternately
  uint32_t * dTileLists[2] = { nullptr, nullptr }; size_t tileListCap[2] = { 0, 0 };
  uint32_t * dTileCounts = nullptr;         // [3][TILE_CLASSES]: recorded by the previous launch | recorded by this one | cleared by this one for the next
  int tileSlot = 0;                         // list set the NEXT launch records into
  int tileCountSlot = 0;                    // count set the NEXT launch records into (zero by then: cleared at creation or by the launch before)
  int tileRecordPeriod = 8;                 // rfx_set_option "tile_order_period": the cost classes are recorded on every k-th launch over a grid; the
                                            // launches in between replay the last recording (no CTA barrier, no atomic at their end: -2 % kernel time)
  int tileReuse = 0;                        // launches that reused the last recording
  bool tileHistory = false;                 // the other set holds the order recorded by the previous launch ...
  uint64_t tileKey[4] = { 0, 0, 0, 0 };     // ... over this grid (image size, row range, strip split)
  bool tileOrdering = true;
  int forcePath = 0;                        // 0 auto, 1 constant bank, 2 blob kernels, 3 blob, general kernel (k_trace_blob_any) only — tests exercise all
  float * dLut = nullptr;
  float4 * dBvhNodes = nullptr; size_t bvhNodesCap = 0;   // big scenes only (see buildBvh)
  int * dBvhPrims = nullptr; size_t bvhPrimsCap = 0;
  int bvhDepth = 0;                         // depth of the hierarchy in dBvhNodes (0: none)
  uint32_t bvhFloat4 = 0;                   // SceneHeader::bvhFloat4 of the uploaded blob
  bool blobSmemBvh = true;                  // rfx_set_option "blob_smem_bvh"
  // shadow-ray candidate grids of the far lights (LightGrid, rfx_types.h): one allocation each for the headers, the cell offsets and the items
  LightGrid * dLightGrids = nullptr; size_t lightGridsCap = 0;
  uint32_t * dGridCells = nullptr; size_t gridCellsCap = 0;
  float4 * dGridSpheres = nullptr; size_t gridSpheresCap = 0;
  int * dGridIndex = nullptr; size_t gridIndexCap = 0;
  bool lightGridsOn = true;                 // rfx_set_option "light_grids"
  // candidate spheres of the first query of a path per 32x32-pixel screen cell (EyeGrid, rfx_kernels.h), rebuilt when the camera,
  // the image size or the scene changes
  uint32_t * dEyeCells = nullptr; size_t eyeCellsCap = 0;
  float4 * dEyeSpheres = nullptr; size_t eyeSpheresCap = 0;
  int * dEyeIndex = nullptr; size_t eyeIndexCap = 0;
  EyeGrid eyeGrid = { nullptr, nullptr, nullptr, 0, 0, 0 };
  uint32_t eyeKey[17] = { 0 }; uint64_t eyeSceneKey = 0; bool eyeValid = false;   // camera (eye, view, rz, wHalf, hHalf as bits) + W, H
  uint64_t sceneUploads = 0;                // bumped by uploadScene
  bool eyeGridOn = true;                    // rfx_set_option "eye_grid"
  uint64_t eyeGridBuilds = 0;
  int lightGridsBuilt = 0;                  // lights of the uploaded scene that have a grid
  int bvhMode = 0;                          // 0 auto (spheres > 32, triangles > 32), 1 always, 2 never — tests compare both
  float4 * dTriNodes = nullptr; size_t triNodesCap = 0;   // hierarchy over the triangles: leaf slots, then pair nodes (uploadScene)
  int * dTriPrims = nullptr; size_t triPrimsCap = 0;
  uint64_t triBvhTris = 0;                  // triangles under that hierarchy in the uploaded scene (0: list walk)

  // ---- camera + render state (reference Render.h:9-27)
  float eye[3] = { 0, 0, 0 }, view[9] = { 1, 0, 0, 0, 1, 0, 0, 0, 1 }, fov = 1.0f;
  uint32_t W = 0, H = 0;
  float * dImage = nullptr; size_t imageCap = 0;
  uint32_t * dSig = nullptr; size_t sigCap = 0; bool sigOn = false;
  int reflNum = 0, sampleNum = 0; bool additive = false; int additiveCounter = 0; bool inProgress = false;
  uint64_t cursor = 0;
  FrameParams snap;           // camera snapshot taken by render_begin

  // ---- random streams
  uint32_t * dRng = nullptr;  // [2] ping-pong LCG state of the Vector3.cpp TU stream
  int rngSlot = 0;
  uint32_t seedRender = 12345u;
  uint32_t * dRngPrefix = nullptr;            // [3][RNG_CLASS_BLOCKS + 1] accept-count prefix sums of the LCG cycle (built at creation)
  RngLocate * dRngLocate = nullptr;
  uint32_t * dSampleStates = nullptr; size_t statesCap = 0;
  uint32_t * dOwnBlocks = nullptr; size_t ownBlocksCap = 0;   // split frames: K1's list of the blocks that hold this GPU's ranks
  int * dStatus = nullptr;
  float * dRays = nullptr; size_t raysCap = 0;   // rfx_trace_rays scratch

  // ---- staging for the host batch path (all slots share one capacity; they are always reallocated together)
  static const int FRAME_SLOTS = 4;
  uint32_t * dFrame[FRAME_SLOTS] = { nullptr, nullptr, nullptr, nullptr }; size_t frameCap = 0;
  uint32_t * dResolve = nullptr; size_t resolveCap = 0;   // K3 output of the Render-API read path (its own buffer and capacity)
  uint64_t maxCallsPerLaunch = 1ull << 25;    // bounds the ranked-state scratch (128 MB) for huge SSAA factors / 8K frames
  float bvhReach[6] = { 0, 0, 0, 0, 0, 0 };   // box of ray origins the hierarchy's margins were sized for (lo xyz, hi xyz)
  float extraOrigins[6] = { FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX };   // box of the ray origins rfx_trace_rays was given
  // path queue of the blob scenes' wavefront kernel pair (rfx_trace_blob.cu): 64-byte records + {count, cursor}
  uint4 * dQueue = nullptr; size_t queueCap = 0;   // in uint4 units (4 per record)
  uint32_t * dQueueCtl = nullptr;
  int blobWavefront = 2;                      // rfx_set_option "blob_wavefront": 0 off, k > 0: the tile kernel of the wavefront renders k segments
  cudaEvent_t evRendered[FRAME_SLOTS] = { nullptr, nullptr, nullptr, nullptr }, evCopied[FRAME_SLOTS] = { nullptr, nullptr, nullptr, nullptr };

  // ---- counters
  unsigned long long * dCounters = nullptr;   // [32][2]
  rfx_stats stats;
  bool profiling = false;
  std::vector<cudaEvent_t> evPool;            // pairs (start, stop) around K2 launches while profiling
  size_t evUsed = 0;
};

namespace
{

int fail(const rfx_ctx * c, int code, const std::string & msg)
{
  if (c) c->err = msg; else g_createError = msg;
  return code;
}

#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return fail(ctx, RFX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
  } while (0)

int useStream(rfx_ctx * ctx, cudaStream_t st)
{
  if (ctx->lastStream && ctx->lastStream != st) CK(cudaStreamSynchronize(ctx->lastStream));
  ctx->lastStream = st;
  return RFX_OK;
}

template <typename T> int ensure(rfx_ctx * ctx, T *& p, size_t & cap, size_t need)
{
  if (need <= cap) return RFX_OK;
  if (p) { CK(cudaDeviceSynchronize()); CK(cudaFree(p)); p = nullptr; cap = 0; }
  const size_t want = need + need / 8;
  CK(cudaMalloc((void **)&p, want * sizeof(T)));
  cap = want;
  return RFX_OK;
}

Material makeMaterial(int mtype, const float rgb[3], float refl, float transp, int order)   // Material.cpp:8-14
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

// flatten the host scene into the blob layout described in rfx_types.h and upload it
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

int uploadScene(rfx_ctx * ctx, cudaStream_t st)
{
  if (!ctx->sceneDirty) return RFX_OK;
  ctx->sceneUploads++;
  ctx->eyeValid = false;

  for (HostTex & t : ctx->tex)
    if (!t.uploaded)
    {
      if (!t.px.empty())
      {
        CK(cudaMalloc((void **)&t.dev, t.px.size() * 4));
        CK(cudaMemcpyAsync(t.dev, t.px.data(), t.px.size() * 4, cudaMemcpyHostToDevice, st));
        ctx->stats.h2d_bytes += t.px.size() * 4;
      }
      t.uploaded = true;
    }

  std::vector<const HostObj *> sph, tri, pla;
  for (const HostObj & o : ctx->objs) (o.kind == 0 ? sph : o.kind == 1 ? tri : pla).push_back(&o);

  SceneHeader h;
  memset(&h, 0, sizeof(h));
  h.nSpheres = (int)sph.size(); h.nTris = (int)tri.size(); h.nPlanes = (int)pla.size();
  h.nLights = (int)ctx->lights.size(); h.nTextures = (int)ctx->tex.size();
  h.skyTex = ctx->skyTex;
  memcpy(h.ambient, ctx->ambient, sizeof(h.ambient));
  h.ambientPower = ctx->ambientPower;
  memcpy(h.env, ctx->env, sizeof(h.env));
  // Skybox::loadTexture / Skybox::Skybox, Skybox.cpp:6-7,21-37
  if (ctx->skyTex >= 0)
  {
    h.halfTileW = (1.0f / 8.0f - 1.0f / float(ctx->tex[ctx->skyTex].w)) - FLT_EPSILON;
    h.halfTileH = (1.0f / 6.0f - 1.0f / float(ctx->tex[ctx->skyTex].h)) - FLT_EPSILON;
  }
  else
  {
    h.halfTileW = 1.0f / 8.0f - FLT_EPSILON;
    h.halfTileH = 1.0f / 6.0f - FLT_EPSILON;
  }
  size_t off = align16(sizeof(SceneHeader));
  h.offLights = (uint32_t)off; off = align16(off + sizeof(Light) * ctx->lights.size());
  h.offSpheres = (uint32_t)off; off = align16(off + sizeof(float) * 4 * sph.size());
  h.offTris = (uint32_t)off; off = align16(off + sizeof(Triangle) * tri.size());
  h.offPlanes = (uint32_t)off; off = align16(off + sizeof(Plane) * pla.size());
  h.offMats = (uint32_t)off; off = align16(off + sizeof(Material) * ctx->objs.size());
  h.offTex = (uint32_t)off; off = align16(off + sizeof(TexRef) * ctx->tex.size());
  // the header addresses the blob with 32-bit offsets (every earlier offset is below off)
  if (off > (size_t)UINT32_MAX) return fail(ctx, RFX_ERR_ARG, "scene too large: the blob exceeds 4 GB");
  h.bytes = (uint32_t)off;
  h.byteLut = ctx->dLut;
  h.bvhPrims = nullptr;
  h.bvhLeafSph = nullptr;
  h.bvhPairs = nullptr;
  h.bvhRoot = 0;
  h.bvhFloat4 = 0;
  h.lightGrids = nullptr;
  ctx->lightGridsBuilt = 0;
  ctx->bvhDepth = 0;
  ctx->bvhFloat4 = 0;
  // automatic mode: more than 32 spheres, and no planes — a drop point on an (unbounded) plane can lie anywhere, so the box margins
  // below, which are sized for ray origins inside a bounded region, could not be guaranteed (the reference's Scene cannot hold
  // planes at all; mode 1 builds the hierarchy regardless, for tests)
  const bool wantBvh = ctx->bvhMode == 1 ? !sph.empty() : ctx->bvhMode == 2 ? false : (sph.size() > 32 && pla.empty());
  // the hierarchy over the triangles: the same automatic rule; mode 1 builds it for any triangle, but never next to a plane (its
  // margins need bounded drop points)
  const bool wantTriBvh = pla.empty() && (ctx->bvhMode == 1 ? !tri.empty() : ctx->bvhMode == 2 ? false : tri.size() > 32);
  ctx->triBvhTris = 0;
  h.triPrims = nullptr; h.triLeaf = nullptr; h.triPairs = nullptr; h.triRoot = 0;
  float lo[3] = { ctx->eye[0], ctx->eye[1], ctx->eye[2] }, hi[3] = { ctx->eye[0], ctx->eye[1], ctx->eye[2] };
  double R = 0.0;
  if (wantBvh || wantTriBvh)
  {
    // Box margins.  The hierarchy must never cull a sphere the reference's exact test (Sphere.cpp:49-57) would report, and that
    // test is noisy: with v = origin - centre, disc = b*b - 4a*c carries an absolute rounding error of at most ~40 * 2^-24 * a|v|^2
    // (three-term dot products, the square, the product), while a ray that misses the sphere by m has disc = 4a(r^2 - m^2).  A
    // "noise hit" therefore needs m^2 - r^2 < 6e-7 |v|^2, i.e. m - r < min(3e-7 |v|^2 / r, 7.7e-4 |v|).  |v| is bounded by the
    // diagonal R of the box that holds every possible ray origin — the camera eye and all drop points (on spheres and
    // triangles) — and every centre; each sphere's box is inflated by twice its own bound, plus 1e-6 R for the device's slab
    // test (fused arithmetic with clamped reciprocals: a box plane moves by at most 2^-22 |origin| along its axis).  (Planes are unbounded: a drop point
    // on a plane can lie outside the box; the reference's Scene cannot hold planes, and rfx_set_camera re-flattens the scene
    // when the eye leaves the box.)
    for (int k = 0; k < 3; k++)
      if (ctx->extraOrigins[k] <= ctx->extraOrigins[3 + k])   // origins of explicit ray lists (rfx_trace_rays)
      {
        lo[k] = std::min(lo[k], ctx->extraOrigins[k]);
        hi[k] = std::max(hi[k], ctx->extraOrigins[3 + k]);
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
    for (int k = 0; k < 3; k++) { ctx->bvhReach[k] = lo[k]; ctx->bvhReach[3 + k] = hi[k]; }
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
      const double noise = std::min(3e-7 * R * R / std::max((double)p.r, 1e-30), 7.7e-4 * R);
      p.m = (float)(2.0 * noise + 1e-6 * R);
      for (int k = 0; k < 3; k++) { p.lo[k] = p.c[k] - p.r - p.m; p.hi[k] = p.c[k] + p.r + p.m; }
    }
    std::vector<BvhNode> nodes;
    int maxDepth = 0;
    buildBvhRec(nodes, prims, 0, (int)prims.size(), 0, maxDepth);
    if (maxDepth <= BLOB_MAX_BVH_DEPTH)   // the traversal stacks hold 24 entries; a median split of 2^20 spheres is 18 deep
    {
      // The device form, one allocation: leaf records — every leaf is 4 slots of (cx, cy, cz, r^2), NaN in the unused ones, so a
      // whole leaf is tested without indirection — then the "pair nodes": an inner node carries both children's boxes,
      // {lo_a.xyz, ref_a} {hi_a.xyz, ref_b} {lo_b.xyz, -} {hi_b.xyz, -}, ref >= 0: pair node index, ref < 0: ~(first slot of a leaf).
      // bvhPrims[4 * leaf + k] = position of that slot's sphere in the sorted sphere array (materials, tie-break order).
      std::vector<int> ref;
      const size_t nLeaves = bvhRefs(nodes, ref);
      const size_t nInner = nodes.size() - nLeaves;
      std::vector<float4> packed(nLeaves * 4 + nInner * 4);
      std::vector<int> order(nLeaves * 4, -1);
      const float qnan = std::numeric_limits<float>::quiet_NaN();
      size_t leaf = 0;
      for (size_t i = 0; i < nodes.size(); i++)
      {
        if (nodes[i].b < 0)
        {
          const int a = nodes[i].a;
          for (int k = 0; k < 4; k++)
          {
            float4 s4 = make_float4(qnan, qnan, qnan, qnan);
            if (k < -nodes[i].b)
            {
              const HostObj * o = sph[prims[a + k].index];
              s4 = make_float4(o->center[0], o->center[1], o->center[2], o->sqRadius);
              order[4 * leaf + k] = prims[a + k].index;
            }
            packed[4 * leaf + k] = s4;
          }
          leaf++;
        }
        else writePairNode(nodes, ref, i, &packed[nLeaves * 4]);
      }
      int rc;
      if ((rc = ensure(ctx, ctx->dBvhNodes, ctx->bvhNodesCap, packed.size())) != RFX_OK) return rc;
      if ((rc = ensure(ctx, ctx->dBvhPrims, ctx->bvhPrimsCap, order.size())) != RFX_OK) return rc;
      CK(cudaMemcpyAsync(ctx->dBvhNodes, packed.data(), packed.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(ctx->dBvhPrims, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      CK(cudaStreamSynchronize(st));
      ctx->stats.h2d_bytes += packed.size() * sizeof(float4) + order.size() * sizeof(int);
      ctx->bvhDepth = maxDepth;
      h.bvhPrims = ctx->dBvhPrims;
      h.bvhLeafSph = ctx->dBvhNodes;
      h.bvhPairs = h.bvhLeafSph + nLeaves * 4;
      h.bvhRoot = ref[0];
      h.bvhFloat4 = (uint32_t)((nLeaves + nInner) * 4);
      ctx->bvhFloat4 = h.bvhFloat4;
      h.bvhRoot = ref[0];

      // shadow-ray candidate grids of the far lights (buildLightGrid).  B: the box of every drop point — all objects (planes are
      // excluded by wantBvh's automatic mode; with planes present no grid is built), padded for the rounding of a drop point
      ctx->lightGridsBuilt = 0;
      if (ctx->lightGridsOn && pla.empty() && !ctx->lights.empty())
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
        std::vector<LightGrid> grids(ctx->lights.size());
        std::vector<uint32_t> cells;
        std::vector<float4> gsph;
        std::vector<int> gidx;
        std::vector<size_t> cellOff(ctx->lights.size(), 0), itemOff(ctx->lights.size(), 0);
        for (size_t li = 0; li < ctx->lights.size(); li++)
        {
          LightGridHost lg;
          memset(&grids[li], 0, sizeof(LightGrid));
          if (!buildLightGrid(ctx->lights[li], sph, prims, blo, bhi, lg)) continue;
          grids[li] = lg.g;
          grids[li].nx = lg.g.nx; grids[li].ny = lg.g.ny;
          cellOff[li] = cells.size(); itemOff[li] = gsph.size();
          cells.insert(cells.end(), lg.cellStart.begin(), lg.cellStart.end());
          gsph.insert(gsph.end(), lg.spheres.begin(), lg.spheres.end());
          gidx.insert(gidx.end(), lg.index.begin(), lg.index.end());
          grids[li].cellStart = reinterpret_cast<const uint32_t *>(1);    // marks "built": patched below once the arrays have their address
          ctx->lightGridsBuilt++;
        }
        if (ctx->lightGridsBuilt)
        {
          if ((rc = ensure(ctx, ctx->dLightGrids, ctx->lightGridsCap, grids.size())) != RFX_OK) return rc;
          if ((rc = ensure(ctx, ctx->dGridCells, ctx->gridCellsCap, cells.size())) != RFX_OK) return rc;
          if ((rc = ensure(ctx, ctx->dGridSpheres, ctx->gridSpheresCap, std::max<size_t>(gsph.size(), 1))) != RFX_OK) return rc;
          if ((rc = ensure(ctx, ctx->dGridIndex, ctx->gridIndexCap, std::max<size_t>(gidx.size(), 1))) != RFX_OK) return rc;
          for (size_t li = 0; li < grids.size(); li++)
            if (grids[li].cellStart)
            {
              grids[li].cellStart = ctx->dGridCells + cellOff[li];
              grids[li].itemSphere = ctx->dGridSpheres + itemOff[li];   // cellStart offsets are relative to the light's own items
              grids[li].itemIndex = ctx->dGridIndex + itemOff[li];
            }
          CK(cudaMemcpyAsync(ctx->dLightGrids, grids.data(), grids.size() * sizeof(LightGrid), cudaMemcpyHostToDevice, st));
          CK(cudaMemcpyAsync(ctx->dGridCells, cells.data(), cells.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
          if (!gsph.empty()) CK(cudaMemcpyAsync(ctx->dGridSpheres, gsph.data(), gsph.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
          if (!gidx.empty()) CK(cudaMemcpyAsync(ctx->dGridIndex, gidx.data(), gidx.size() * sizeof(int), cudaMemcpyHostToDevice, st));
          CK(cudaStreamSynchronize(st));
          ctx->stats.h2d_bytes += grids.size() * sizeof(LightGrid) + cells.size() * 4 + gsph.size() * 16 + gidx.size() * 4;
          h.lightGrids = ctx->dLightGrids;
        }
      }
    }
  }
  if (wantTriBvh)
  {
    // The hierarchy over the triangles (buildTriBoxes has the boxes and their margins).  Device form, one allocation: leaf slots of
    // 3 float4 each (4 per leaf, the layout of SmallScene::triPk; unused slots all zero, which the exact test's gate |rz| > 2^-63
    // rejects), then the pair nodes; triPrims[slot] = the slot's position in the sorted triangle array (-1 unused).
    std::vector<float> tv(tri.size() * 12), boxes(tri.size() * 6);
    for (size_t i = 0; i < tri.size(); i++) { memcpy(&tv[12 * i], tri[i]->tri.v0, 12); memcpy(&tv[12 * i + 3], tri[i]->tri.ax, 36); }
    buildTriBoxes((int)tri.size(), tv.data(), ctx->bvhReach, boxes.data());
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
      std::vector<int> ref;
      const size_t nLeaves = bvhRefs(nodes, ref), nInner = nodes.size() - nLeaves;
      std::vector<float4> packed(nLeaves * 12 + nInner * 4, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
      std::vector<int> order(nLeaves * 4, -1);
      size_t leaf = 0;
      for (size_t i = 0; i < nodes.size(); i++)
      {
        if (nodes[i].b < 0)
        {
          for (int k = 0; k < -nodes[i].b; k++)
          {
            const int ti = prims[nodes[i].a + k].index;
            const Triangle & t = tri[ti]->tri;
            float4 * w = &packed[12 * leaf + 3 * k];
            w[0] = make_float4(t.v0[0], t.v0[1], t.v0[2], t.ax[6]);
            w[1] = make_float4(t.ax[7], t.ax[8], t.ax[0], t.ax[1]);
            w[2] = make_float4(t.ax[2], t.ax[3], t.ax[4], t.ax[5]);
            order[4 * leaf + k] = ti;
          }
          leaf++;
        }
        else writePairNode(nodes, ref, i, &packed[nLeaves * 12]);
      }
      int rc;
      if ((rc = ensure(ctx, ctx->dTriNodes, ctx->triNodesCap, packed.size())) != RFX_OK) return rc;
      if ((rc = ensure(ctx, ctx->dTriPrims, ctx->triPrimsCap, order.size())) != RFX_OK) return rc;
      CK(cudaMemcpyAsync(ctx->dTriNodes, packed.data(), packed.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(ctx->dTriPrims, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice, st));
      CK(cudaStreamSynchronize(st));
      ctx->stats.h2d_bytes += packed.size() * sizeof(float4) + order.size() * sizeof(int);
      h.triPrims = ctx->dTriPrims;
      h.triLeaf = ctx->dTriNodes;
      h.triPairs = ctx->dTriNodes + nLeaves * 12;
      h.triRoot = ref[0];
      ctx->triBvhTris = tri.size();
    }
  }

  std::vector<unsigned char> blob(off, 0);
  memcpy(blob.data(), &h, sizeof(h));
  if (!ctx->lights.empty()) memcpy(blob.data() + h.offLights, ctx->lights.data(), sizeof(Light) * ctx->lights.size());
  Material * mats = reinterpret_cast<Material *>(blob.data() + h.offMats);
  size_t mi = 0;
  for (size_t i = 0; i < sph.size(); i++)
  {
    float * d = reinterpret_cast<float *>(blob.data() + h.offSpheres) + 4 * i;
    d[0] = sph[i]->center[0]; d[1] = sph[i]->center[1]; d[2] = sph[i]->center[2]; d[3] = sph[i]->sqRadius;
    mats[mi++] = sph[i]->mat;
  }
  for (size_t i = 0; i < tri.size(); i++)
  {
    reinterpret_cast<Triangle *>(blob.data() + h.offTris)[i] = tri[i]->tri;
    mats[mi++] = tri[i]->mat;
  }
  for (size_t i = 0; i < pla.size(); i++)
  {
    reinterpret_cast<Plane *>(blob.data() + h.offPlanes)[i] = pla[i]->plane;
    mats[mi++] = pla[i]->mat;
  }
  for (size_t i = 0; i < ctx->tex.size(); i++)
  {
    TexRef r;
    r.px = ctx->tex[i].dev; r.w = ctx->tex[i].w; r.h = ctx->tex[i].h;
    reinterpret_cast<TexRef *>(blob.data() + h.offTex)[i] = r;
  }

  if (off > ctx->blobCap)
  {
    if (ctx->dBlob) { CK(cudaDeviceSynchronize()); CK(cudaFree(ctx->dBlob)); ctx->dBlob = nullptr; }
    CK(cudaMalloc((void **)&ctx->dBlob, off));
    ctx->blobCap = off;
  }
  // pageable source: the copy is staged before the call returns, so the local vector may die
  CK(cudaMemcpyAsync(ctx->dBlob, blob.data(), off, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  ctx->stats.h2d_bytes += off;
  ctx->blobBytes = (uint32_t)off;

  // constant-bank form (rfx_trace_small.cu)
  ctx->smallOk = sph.size() <= (size_t)SMALL_MAX_SPHERES && tri.size() <= (size_t)SMALL_MAX_TRIS && pla.size() <= (size_t)SMALL_MAX_PLANES &&
                 ctx->lights.size() <= (size_t)SMALL_MAX_LIGHTS && ctx->tex.size() <= (size_t)SMALL_MAX_TEX;
  if (ctx->smallOk)
  {
    SmallScene & ss = ctx->small;
    memset(&ss, 0, sizeof(ss));
    ss.nS = h.nSpheres; ss.nT = h.nTris; ss.nP = h.nPlanes; ss.nL = h.nLights;
    ss.skyTex = h.skyTex; ss.halfTileW = h.halfTileW; ss.halfTileH = h.halfTileH;
    ss.ambientPower = h.ambientPower;
    memcpy(ss.ambient, h.ambient, sizeof(ss.ambient));
    memcpy(ss.env, h.env, sizeof(ss.env));
    ss.byteLut = ctx->dLut;
    for (size_t i = 0; i < sph.size(); i++)
    {
      ss.sph[i] = make_float4(sph[i]->center[0], sph[i]->center[1], sph[i]->center[2], sph[i]->sqRadius);
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
      const Triangle & t = tri[i]->tri;
      ss.tri[i] = t; ss.mat[SMALL_MAX_SPHERES + i] = tri[i]->mat;
      ss.triPk[i][0] = make_float4(t.v0[0], t.v0[1], t.v0[2], t.ax[6]);
      ss.triPk[i][1] = make_float4(t.ax[7], t.ax[8], t.ax[0], t.ax[1]);
      ss.triPk[i][2] = make_float4(t.ax[2], t.ax[3], t.ax[4], t.ax[5]);
    }
    for (size_t i = 0; i < pla.size(); i++) { ss.pl[i] = pla[i]->plane; ss.mat[SMALL_MAX_SPHERES + SMALL_MAX_TRIS + i] = pla[i]->mat; }
    for (size_t i = 0; i < ctx->lights.size(); i++) ss.light[i] = ctx->lights[i];
    for (size_t i = 0; i < ctx->tex.size(); i++) { ss.tex[i].px = ctx->tex[i].dev; ss.tex[i].w = ctx->tex[i].w; ss.tex[i].h = ctx->tex[i].h; }
  }
  ctx->sceneDirty = false;
  return RFX_OK;
}

// number of block-preview origins (x % a == 0 && y % a == 0) with linear index < p, scan order
uint64_t originsBefore(uint64_t p, uint32_t W, uint32_t a)
{
  const uint64_t bw = (W + a - 1) / a;
  const uint64_t y = p / W, x = p % W;
  uint64_t n = ((y + a - 1) / a) * bw;            // complete origin rows below y
  if (y % a == 0) n += (x + a - 1) / a;           // origins left of x in this row
  return n;
}

// rank n Scene::trace calls on the randDir stream; the states land in ctx->dSampleStates (or nowhere when skipOnly)
int rankSamples(rfx_ctx * ctx, uint64_t n, bool skipOnly, cudaStream_t st, uint64_t ownPeriod = 0, uint32_t ownWorld = 0, uint32_t ownRank = 0)
{
  if (n == 0) return RFX_OK;
  const uint32_t nBlocks = rngBlocksFor(n);
  int rc;
  if (!skipOnly && (rc = ensure(ctx, ctx->dSampleStates, ctx->statesCap, n)) != RFX_OK) return rc;
  RngWork w;
  w.stateIn = ctx->dRng + ctx->rngSlot;
  w.stateOut = ctx->dRng + (ctx->rngSlot ^ 1);
  w.prefix = ctx->dRngPrefix;
  w.locate = ctx->dRngLocate;
  w.sampleStates = skipOnly ? nullptr : ctx->dSampleStates;
  w.status = ctx->dStatus;
  w.n = n;
  w.nBlocks = nBlocks;
  w.ownPeriod = ownPeriod; w.ownWorld = ownWorld; w.ownRank = ownRank;
  if (ownWorld && !skipOnly)
  {
    const uint32_t bound = rngOwnBlocksBound(n, ownPeriod, ownWorld, nBlocks);
    if ((rc = ensure(ctx, ctx->dOwnBlocks, ctx->ownBlocksCap, bound)) != RFX_OK) return rc;
    w.ownList = ctx->dOwnBlocks; w.ownListCap = (uint32_t)std::min<size_t>(ctx->ownBlocksCap, 0xFFFFFFFFu);
  }
  ctx->stats.kernel_launches += launchRngRank(w, st);
  CK(cudaGetLastError());
  ctx->rngSlot ^= 1;
  return RFX_OK;
}

// Fills w.order for a fast-kernel launch and remembers what the launch will have recorded (see TileOrder).  History is
// only reused by a launch over exactly the same grid; any other launch of the fast kernel starts a new history.
// ---- candidates of the first query of a path (EyeGrid) ------------------------------------------------------------------------------
// Scenes with a sphere hierarchy: every path starts at the eye, so the spheres its first query can hit are the ones whose primary-ray
// screen bounds (primarySphereBounds: the rectangles the constant-bank kernel's tiles use, conservative against the float noise of
// the exact test, SSAA sub-samples and jitter) cover its pixel.  The host bins the rectangles into 32x32-pixel cells per camera; a
// 4x8 tile lies in one cell, so its 32 lanes walk the same short list instead of the hierarchy.  Closest hit over a complete
// candidate list is the hierarchy walk's answer (ties go to the lower insertion index in both).
constexpr int EYE_GRID_SHIFT = 5;      // 32x32-pixel cells: a 4x8 tile of the kernels lies in one cell

// the binning itself, a pure function (rfx_selftest_eye_grid_host checks it on the CPU): spheres[i] = (cx, cy, cz, r^2)
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

int buildEyeGrid(rfx_ctx * ctx, const FrameParams & fp, cudaStream_t st)
{
  ctx->eyeGrid.cellStart = nullptr;
  if (!ctx->eyeGridOn || ctx->bvhDepth <= 0) return RFX_OK;
  uint32_t key[17];
  memcpy(key, fp.eye, 12); memcpy(key + 3, fp.view, 36);
  memcpy(key + 12, &fp.rz, 4); memcpy(key + 13, &fp.wHalf, 4); memcpy(key + 14, &fp.hHalf, 4);
  key[15] = fp.W; key[16] = fp.H;
  if (ctx->eyeValid && ctx->eyeSceneKey == ctx->sceneUploads && !memcmp(key, ctx->eyeKey, sizeof(key)))
  {
    ctx->eyeGrid.cellStart = ctx->dEyeCells;
    return RFX_OK;
  }
  ctx->eyeValid = false;
  std::vector<float4> spheres;       // in the order of the sorted sphere array (uploadScene walks the objects the same way)
  for (const HostObj & o : ctx->objs) if (o.kind == 0) spheres.push_back(make_float4(o.center[0], o.center[1], o.center[2], o.sqRadius));
  int nx = 0, ny = 0;
  std::vector<uint32_t> cells;
  std::vector<float4> items;
  std::vector<int> index;
  if (!binEyeGrid(fp, spheres, nx, ny, cells, items, index)) return RFX_OK;
  int rc;
  if ((rc = ensure(ctx, ctx->dEyeCells, ctx->eyeCellsCap, cells.size())) != RFX_OK) return rc;
  if ((rc = ensure(ctx, ctx->dEyeSpheres, ctx->eyeSpheresCap, items.size())) != RFX_OK) return rc;
  if ((rc = ensure(ctx, ctx->dEyeIndex, ctx->eyeIndexCap, index.size())) != RFX_OK) return rc;
  // pageable sources: each copy is staged before its call returns, and the copies are ordered on the stream behind the kernels of
  // the previous frame that still read the old grid
  CK(cudaMemcpyAsync(ctx->dEyeCells, cells.data(), cells.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->dEyeSpheres, items.data(), items.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->dEyeIndex, index.data(), index.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  ctx->stats.h2d_bytes += cells.size() * 4 + items.size() * 16 + index.size() * 4;
  ctx->eyeGrid.cellStart = ctx->dEyeCells; ctx->eyeGrid.itemSphere = ctx->dEyeSpheres; ctx->eyeGrid.itemIndex = ctx->dEyeIndex;
  ctx->eyeGrid.nx = nx; ctx->eyeGrid.ny = ny; ctx->eyeGrid.shift = EYE_GRID_SHIFT;
  memcpy(ctx->eyeKey, key, sizeof(key)); ctx->eyeSceneKey = ctx->sceneUploads; ctx->eyeValid = true;
  ctx->eyeGridBuilds++;
  return RFX_OK;
}

int armTileOrder(rfx_ctx * ctx, TraceWork & w, cudaStream_t st)
{
  w.order = TileOrder();
  const uint32_t grid = ctx->smallOk && ctx->forcePath < 2 ? fastGridSize(w) : 0;
  if (!ctx->tileOrdering || grid == 0 || grid > (1u << 22)) { ctx->tileHistory = false; return RFX_OK; }
  const uint64_t key[4] = { ((uint64_t)w.fp.W << 32) | w.fp.H, w.fp.p0, w.fp.p1,
                            ((uint64_t)w.fp.stripRows << 40) | ((uint64_t)w.fp.stripWorld << 20) | w.fp.stripRank };
  int rc;
  const int out = ctx->tileSlot, in = out ^ 1;
  const int cOut = ctx->tileCountSlot, cIn = (cOut + 2) % 3, cNext = (cOut + 1) % 3;
  if (ctx->tileRecordPeriod > 1 && ctx->tileHistory && memcmp(key, ctx->tileKey, sizeof(key)) == 0 && ctx->tileReuse + 1 < ctx->tileRecordPeriod &&
      ctx->tileListCap[in] >= (size_t)grid * TILE_CLASSES)
  {
    // replay the last recording without recording again (the kernel then has no CTA barrier and no atomic at its end)
    w.order.inLists = ctx->dTileLists[in];
    w.order.inCounts = ctx->dTileCounts + cIn * TILE_CLASSES;
    w.order.capacity = grid;
    ctx->tileReuse++;
    return RFX_OK;
  }
  ctx->tileReuse = 0;
  if ((rc = ensure(ctx, ctx->dTileLists[out], ctx->tileListCap[out], (size_t)grid * TILE_CLASSES)) != RFX_OK) return rc;
  if (!ctx->dTileCounts)
  {
    CK(cudaMalloc((void **)&ctx->dTileCounts, 3 * TILE_CLASSES * sizeof(uint32_t)));
    CK(cudaMemsetAsync(ctx->dTileCounts, 0, 3 * TILE_CLASSES * sizeof(uint32_t), st));
  }
  w.order.outLists = ctx->dTileLists[out];
  w.order.outCounts = ctx->dTileCounts + cOut * TILE_CLASSES;
  w.order.zeroCounts = ctx->dTileCounts + cNext * TILE_CLASSES;
  w.order.capacity = grid;
  if (ctx->tileHistory && memcmp(key, ctx->tileKey, sizeof(key)) == 0 && ctx->tileListCap[in] >= (size_t)grid * TILE_CLASSES)
  {
    w.order.inLists = ctx->dTileLists[in];
    w.order.inCounts = ctx->dTileCounts + cIn * TILE_CLASSES;
  }
  ctx->tileCountSlot = cNext;
  memcpy(ctx->tileKey, key, sizeof(key));
  ctx->tileHistory = true;
  ctx->tileSlot = in;
  return RFX_OK;
}

// render pixels [p0, p1) of the frame latched by render_begin
// preStates: random states already ranked for exactly [p0, p1) (batch path ranks several frames per K1 pass); NULL = rank here
int renderRange(rfx_ctx * ctx, uint64_t p0, uint64_t p1, uint32_t * argbOut, bool writeImage, cudaStream_t st,
                const uint32_t * preStates = nullptr)
{
  int rc;
  const int sn = ctx->sampleNum;
  uint64_t cur = p0;
  while (cur < p1)
  {
    uint64_t end, nCalls, firstRank = 0;
    if (sn > 0)
    {
      const uint64_t per = (uint64_t)sn * sn;
      uint64_t pix = ctx->maxCallsPerLaunch / per;
      if (pix < 1) pix = 1;
      if (cur % ctx->W == 0 && pix >= ctx->W) pix -= pix % ctx->W;   // whole rows keep the chunk on the tiled fast kernel
      end = preStates ? p1 : std::min(p1, cur + pix);
      nCalls = (end - cur) * per;
    }
    else
    {
      const uint32_t a = (uint32_t)(-sn);
      end = p1;   // at most one call per a*a pixels: never exceeds the cap for any sane image
      firstRank = originsBefore(cur, ctx->W, a);
      nCalls = originsBefore(end, ctx->W, a) - firstRank;
    }
    if (nCalls > 0)
    {
      if (!preStates && (rc = rankSamples(ctx, nCalls, false, st)) != RFX_OK) return rc;
      TraceWork w;
      w.sceneBlob = ctx->dBlob;
      w.sceneBytes = ctx->blobBytes;
      w.fp = ctx->snap;
      w.fp.p0 = cur; w.fp.p1 = end; w.fp.firstRank = firstRank;
      w.fp.seedRender = ctx->seedRender;
      w.sampleStates = preStates ? preStates : ctx->dSampleStates;
      w.image = writeImage ? ctx->dImage : nullptr;
      w.argbOut = argbOut;
      w.sigOut = ctx->sigOn ? ctx->dSig : nullptr;
      w.counters = ctx->dCounters;
      w.lightGrids = ctx->lightGridsBuilt > 0;
      w.triBvh = ctx->triBvhTris > 0;
      cudaEvent_t evA = nullptr, evB = nullptr;
      if (ctx->profiling)
      {
        if (ctx->evUsed + 2 > ctx->evPool.size())
          for (int i = 0; i < 2; i++) { cudaEvent_t e; CK(cudaEventCreate(&e)); ctx->evPool.push_back(e); }
        evA = ctx->evPool[ctx->evUsed++]; evB = ctx->evPool[ctx->evUsed++];
        CK(cudaEventRecord(evA, st));
      }
      const bool useSmall = ctx->forcePath >= 2 ? false : ctx->smallOk;
      if (useSmall && (rc = armTileOrder(ctx, w, st)) != RFX_OK) return rc;
      if (useSmall)
      {
        uint32_t fastGrid = 0;
        const int nl = launchTraceSmall(ctx->small, w, st, &fastGrid);
        ctx->stats.kernel_launches += nl;
        (fastGrid ? ctx->stats.launches_small_fast : ctx->stats.launches_small_any) += nl;
      }
      else
      {
        const uint64_t wavePixels = (ctx->blobWavefront && ctx->forcePath != 3) ? blobWavePixels(w) : 0;
        if (wavePixels)
        {
          if ((rc = ensure(ctx, ctx->dQueue, ctx->queueCap, (size_t)wavePixels * 4)) != RFX_OK) return rc;   // 64-byte records
          if (!ctx->dQueueCtl) CK(cudaMalloc((void **)&ctx->dQueueCtl, 2 * sizeof(uint32_t)));
        }
        if ((rc = buildEyeGrid(ctx, w.fp, st)) != RFX_OK) return rc;
        w.eyeGrid = ctx->eyeGrid;
        int nl = ctx->forcePath == 3 ? 0 : launchTraceBlobFast(w, st, wavePixels ? ctx->dQueue : nullptr, ctx->dQueueCtl, (uint32_t)ctx->prop.multiProcessorCount * 8u,
                                                               ctx->blobWavefront, ctx->blobSmemBvh ? ctx->bvhFloat4 : 0u);
        if (nl) ctx->stats.launches_blob_fast += nl;
        else { nl = launchTraceBlobAny(w, st); ctx->stats.launches_blob_any += nl; }
        ctx->stats.kernel_launches += nl;
      }
      if (evB) CK(cudaEventRecord(evB, st));
      CK(cudaGetLastError());
      ctx->stats.samples += nCalls;
      if (ctx->snap.jitter && sn > 0) ctx->seedRender = lcgJumpHost(ctx->seedRender, 2 * (end - cur));
    }
    cur = end;
  }
  return RFX_OK;
}

int checkStatus(rfx_ctx * ctx)
{
  int status = 0;
  CK(cudaMemcpy(&status, ctx->dStatus, sizeof(int), cudaMemcpyDeviceToHost));
  if (status) return fail(ctx, RFX_ERR_RNG, "random-stream ranking ran out of over-provisioned draws");
  return RFX_OK;
}

} // namespace

// =====================================================================================================================
extern "C"
{

const char * rfx_version(void) { return "reflaxman_b200 0.1 (sm_100a)"; }

int rfx_create(rfx_ctx ** out, int device)
{
  rfx_ctx * ctx = nullptr;   // for CK
  if (!out) return fail(nullptr, RFX_ERR_ARG, "rfx_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(nullptr, RFX_ERR_NODEV, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(nullptr, RFX_ERR_ARG, "rfx_create: bad device ordinal");
  cudaDeviceProp prop;
  CK(cudaSetDevice(device));
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(nullptr, RFX_ERR_NODEV, std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                ", this library carries sm_100a code only (there is no CPU fallback)");
  ctx = new rfx_ctx();
  ctx->device = device;
  ctx->prop = prop;
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  memset(&ctx->snap, 0, sizeof(ctx->snap));
  cudaError_t err = cudaSuccess;
  auto step = [&](cudaError_t r) { if (err == cudaSuccess) err = r; };
  step(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) step(cudaStreamCreateWithFlags(&ctx->copyStream[i], cudaStreamNonBlocking));
  if (initRngTables() != 0) step(cudaErrorUnknown);
  step(cudaMalloc((void **)&ctx->dRng, 2 * sizeof(uint32_t)));
  step(cudaMalloc((void **)&ctx->dRngPrefix, 3 * (size_t)(RNG_CLASS_BLOCKS + 1) * sizeof(uint32_t)));
  step(cudaMalloc((void **)&ctx->dRngLocate, sizeof(RngLocate)));
  if (err == cudaSuccess)
  {
    // accept counts of the whole LCG cycle: ~5 ms once per context; every later ranking or skip is a table lookup away
    uint32_t * counts = nullptr;
    step(cudaMalloc((void **)&counts, 3 * (size_t)RNG_CLASS_BLOCKS * sizeof(uint32_t)));
    if (err == cudaSuccess) { launchRngTable(counts, ctx->dRngPrefix, ctx->stream); step(cudaStreamSynchronize(ctx->stream)); step(cudaGetLastError()); }
    cudaFree(counts);
  }
  step(cudaMalloc((void **)&ctx->dStatus, sizeof(int)));
  step(cudaMalloc((void **)&ctx->dCounters, 64 * sizeof(unsigned long long)));
  step(cudaMalloc((void **)&ctx->dLut, 256 * sizeof(float)));
  for (int i = 0; i < rfx_ctx::FRAME_SLOTS; i++)
  {
    step(cudaEventCreateWithFlags(&ctx->evRendered[i], cudaEventDisableTiming));
    step(cudaEventCreateWithFlags(&ctx->evCopied[i], cudaEventDisableTiming));
  }
  if (err == cudaSuccess)
  {
    float lut[256];
    for (int i = 0; i < 256; i++) lut[i] = float(i) / 255.0f;   // Color(ARGB), Color.cpp:11-13
    const uint32_t seeds[2] = { 12345u, 12345u };
    step(cudaMemcpy(ctx->dLut, lut, sizeof(lut), cudaMemcpyHostToDevice));
    step(cudaMemcpy(ctx->dRng, seeds, sizeof(seeds), cudaMemcpyHostToDevice));
    step(cudaMemset(ctx->dStatus, 0, sizeof(int)));
    step(cudaMemset(ctx->dCounters, 0, 64 * sizeof(unsigned long long)));
  }
  if (err != cudaSuccess)
  {
    std::string msg = std::string("rfx_create: ") + cudaGetErrorString(err);
    rfx_destroy(ctx);
    return fail(nullptr, RFX_ERR_CUDA, msg);
  }
  *out = ctx;
  return RFX_OK;
}

void rfx_destroy(rfx_ctx * ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (HostTex & t : ctx->tex) if (t.dev) cudaFree(t.dev);
  cudaFree(ctx->dBlob); cudaFree(ctx->dLut); cudaFree(ctx->dImage); cudaFree(ctx->dSig); cudaFree(ctx->dRng);
  cudaFree(ctx->dRngPrefix); cudaFree(ctx->dRngLocate); cudaFree(ctx->dSampleStates); cudaFree(ctx->dStatus);
  cudaFree(ctx->dCounters); cudaFree(ctx->dRays); cudaFree(ctx->dBvhNodes); cudaFree(ctx->dBvhPrims); cudaFree(ctx->dTriNodes); cudaFree(ctx->dTriPrims); cudaFree(ctx->dEyeCells); cudaFree(ctx->dEyeSpheres); cudaFree(ctx->dEyeIndex); cudaFree(ctx->dLightGrids); cudaFree(ctx->dGridCells); cudaFree(ctx->dGridSpheres); cudaFree(ctx->dGridIndex); cudaFree(ctx->dTileLists[0]); cudaFree(ctx->dTileLists[1]); cudaFree(ctx->dTileCounts);
  for (cudaEvent_t e : ctx->evPool) cudaEventDestroy(e);
  cudaFree(ctx->dResolve); cudaFree(ctx->dQueue); cudaFree(ctx->dQueueCtl); cudaFree(ctx->dOwnBlocks);
  for (int i = 0; i < rfx_ctx::FRAME_SLOTS; i++)
  {
    cudaFree(ctx->dFrame[i]);
    if (ctx->evRendered[i]) cudaEventDestroy(ctx->evRendered[i]);
    if (ctx->evCopied[i]) cudaEventDestroy(ctx->evCopied[i]);
  }
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  for (int i = 0; i < 2; i++) if (ctx->copyStream[i]) cudaStreamDestroy(ctx->copyStream[i]);
  delete ctx;
}

const char * rfx_last_error(const rfx_ctx * ctx) { return ctx ? ctx->err.c_str() : g_createError.c_str(); }

int rfx_get_device_info(const rfx_ctx * ctx, rfx_device_info * out)
{
  if (!ctx || !out) return RFX_ERR_ARG;
  memset(out, 0, sizeof(*out));
  out->device = ctx->device;
  out->sm_count = ctx->prop.multiProcessorCount;
  out->cc_major = ctx->prop.major; out->cc_minor = ctx->prop.minor;
  int khz = 0;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
  out->clock_khz = khz;
  out->total_mem = ctx->prop.totalGlobalMem;
  strncpy(out->name, ctx->prop.name, sizeof(out->name) - 1);
  return RFX_OK;
}

// ---------------------------------------------------------------------------------------------------------- scene
int rfx_scene_reset(rfx_ctx * ctx, const float ambient_rgb[3], float ambient_power)
{
  if (!ctx || !ambient_rgb) return fail(ctx, RFX_ERR_ARG, "rfx_scene_reset: NULL argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  for (HostTex & t : ctx->tex) if (t.dev) cudaFree(t.dev);
  ctx->tex.clear(); ctx->objs.clear(); ctx->lights.clear();
  ctx->skyTex = -1;
  for (int i = 0; i < 3; i++) { ctx->extraOrigins[i] = FLT_MAX; ctx->extraOrigins[3 + i] = -FLT_MAX; }
  for (int i = 0; i < 3; i++)
  {
    ctx->ambient[i] = ambient_rgb[i];
    ctx->env[i] = ambient_rgb[i] * ambient_power;   // envColor(diffLightColor * diffLightPower), Scene.cpp:12
  }
  ctx->ambientPower = ambient_power;
  ctx->sceneDirty = true;
  return RFX_OK;
}

int rfx_add_light(rfx_ctx * ctx, const float o[3], float radius, const float rgb[3], float power)
{
  if (!ctx || !o || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_light: NULL argument");
  if (radius <= VSN) radius = VSN;                              // Scene.cpp:51-52
  for (int i = 0; i < 3; i++) ctx->env[i] = ctx->env[i] + rgb[i] * power;   // envColor += color * power, Scene.cpp:54
  Light l;
  l.ox = o[0]; l.oy = o[1]; l.oz = o[2]; l.radius = radius;
  l.r = rgb[0]; l.g = rgb[1]; l.b = rgb[2];
  l.power = clampf(power, 0.0f, 1.0f);                          // OmniLight.cpp:13
  ctx->lights.push_back(l);
  ctx->sceneDirty = true;
  return (int)ctx->lights.size() - 1;
}

int rfx_add_sphere(rfx_ctx * ctx, const float c[3], float radius, int mtype, const float rgb[3], float refl, float transp)
{
  if (!ctx || !c || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_sphere: NULL argument");
  if (radius <= VSN) radius = VSN;                              // Scene.cpp:33-34
  HostObj o;
  memset(&o, 0, sizeof(o));
  o.kind = 0;
  o.mat = makeMaterial(mtype, rgb, refl, transp, (int)ctx->objs.size());
  o.center[0] = c[0]; o.center[1] = c[1]; o.center[2] = c[2];
  o.sqRadius = radius * radius;                                 // Sphere.cpp:19
  o.radius = radius;
  ctx->objs.push_back(o);
  ctx->sceneDirty = true;
  return (int)ctx->objs.size() - 1;
}

int rfx_add_triangle(rfx_ctx * ctx, const float v[9], int mtype, const float rgb[3], float refl, float transp)
{
  if (!ctx || !v || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_triangle: NULL argument");
  HostObj o;
  memset(&o, 0, sizeof(o));
  o.kind = 1;
  o.mat = makeMaterial(mtype, rgb, refl, transp, (int)ctx->objs.size());
  const H3 v0 = { v[0], v[1], v[2] }, v1 = { v[3], v[4], v[5] }, v2 = { v[6], v[7], v[8] };
  const H3 n = hnormalize(hcross(hsub(v1, v0), hsub(v2, v0)));  // Triangle.cpp:13
  const H3 nn = { -n.x, -n.y, -n.z };
  invertColumns(hsub(v2, v0), hsub(v1, v0), nn, o.tri.ax);      // Triangle.cpp:19-20
  o.tri.v0[0] = v0.x; o.tri.v0[1] = v0.y; o.tri.v0[2] = v0.z;
  o.tri.n[0] = n.x; o.tri.n[1] = n.y; o.tri.n[2] = n.z;
  memcpy(o.triVerts, v, sizeof(o.triVerts));
  ctx->objs.push_back(o);
  ctx->sceneDirty = true;
  return (int)ctx->objs.size() - 1;
}

int rfx_add_mesh(rfx_ctx * ctx, uint32_t n_vertices, const float * xyz, uint32_t n_tris, const uint32_t * idx, int mtype, const float rgb[3],
                 float refl, float transp)
{
  if (!ctx || !xyz || !idx || !rgb || n_tris == 0) return fail(ctx, RFX_ERR_ARG, "rfx_add_mesh: NULL argument or no triangle");
  if ((uint64_t)ctx->objs.size() + n_tris > (uint64_t)INT32_MAX) return fail(ctx, RFX_ERR_ARG, "rfx_add_mesh: too many objects");
  for (uint64_t k = 0; k < 3ull * n_tris; k++)
    if (idx[k] >= n_vertices) return fail(ctx, RFX_ERR_ARG, "rfx_add_mesh: vertex index out of range");
  const int first = (int)ctx->objs.size();
  ctx->objs.reserve(ctx->objs.size() + n_tris);
  for (uint32_t k = 0; k < n_tris; k++)
  {
    float v[9];
    for (int j = 0; j < 3; j++) memcpy(v + 3 * j, xyz + 3 * (size_t)idx[3 * (size_t)k + j], 12);
    const int rc = rfx_add_triangle(ctx, v, mtype, rgb, refl, transp);
    if (rc < 0) return rc;
  }
  return first;
}

int rfx_set_triangle_texture(rfx_ctx * ctx, int object, int texture, const float uv[6])
{
  if (!ctx || !uv) return fail(ctx, RFX_ERR_ARG, "rfx_set_triangle_texture: NULL argument");
  if (object < 0 || object >= (int)ctx->objs.size() || ctx->objs[object].kind != 1)
    return fail(ctx, RFX_ERR_ARG, "rfx_set_triangle_texture: object is not a triangle");
  if (texture < 0 || texture >= (int)ctx->tex.size()) return fail(ctx, RFX_ERR_ARG, "rfx_set_triangle_texture: unknown texture");
  HostObj & o = ctx->objs[object];
  // tuvTrans = Matrix33(v3 - v1, v2 - v1, (0,0,-1)) with v_i = (tu_i, tv_i, 0), Triangle.cpp:116-119
  o.tri.tuv[0] = uv[4] - uv[0]; o.tri.tuv[1] = uv[2] - uv[0];
  o.tri.tuv[2] = uv[5] - uv[1]; o.tri.tuv[3] = uv[3] - uv[1];
  o.tri.tu0 = uv[0]; o.tri.tv0 = uv[1];
  o.mat.tex = texture;
  ctx->sceneDirty = true;
  return RFX_OK;
}

int rfx_add_plane(rfx_ctx * ctx, const float pos[3], const float norm[3], int mtype, const float rgb[3], float refl, float transp)
{
  if (!ctx || !pos || !norm || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_plane: NULL argument");
  HostObj o;
  memset(&o, 0, sizeof(o));
  o.kind = 2;
  o.mat = makeMaterial(mtype, rgb, refl, transp, (int)ctx->objs.size());
  memcpy(o.plane.pos, pos, sizeof(float) * 3);
  memcpy(o.plane.n, norm, sizeof(float) * 3);
  ctx->objs.push_back(o);
  ctx->sceneDirty = true;
  return (int)ctx->objs.size() - 1;
}

int rfx_add_texture_argb(rfx_ctx * ctx, uint32_t w, uint32_t h, const uint32_t * argb)
{
  if (!ctx) return RFX_ERR_ARG;
  HostTex t;
  if (argb && w && h)
  {
    t.w = w; t.h = h;
    t.px.assign(argb, argb + (size_t)w * h);
  }
  ctx->tex.push_back(std::move(t));
  ctx->sceneDirty = true;
  return (int)ctx->tex.size() - 1;
}

int rfx_set_skybox(rfx_ctx * ctx, int texture)
{
  if (!ctx) return RFX_ERR_ARG;
  if (texture >= (int)ctx->tex.size()) return fail(ctx, RFX_ERR_ARG, "rfx_set_skybox: unknown texture");
  // Skybox::loadTexture returns false and keeps the checker when the file failed to load (Skybox.cpp:30-36)
  ctx->skyTex = (texture >= 0 && !ctx->tex[texture].px.empty()) ? texture : -1;
  ctx->sceneDirty = true;
  return ctx->skyTex >= 0 ? 1 : 0;
}

// --------------------------------------------------------------------------------------------------------- camera
int rfx_set_camera(rfx_ctx * ctx, const float eye[3], const float view[9], float fov)
{
  if (!ctx || !eye || !view) return fail(ctx, RFX_ERR_ARG, "rfx_set_camera: NULL argument");
  memcpy(ctx->eye, eye, sizeof(float) * 3);
  memcpy(ctx->view, view, sizeof(float) * 9);
  ctx->fov = fov;
  // the hierarchies' box margins were sized for ray origins inside bvhReach (uploadScene): an eye outside it re-flattens the scene
  if (ctx->bvhDepth > 0 || ctx->triBvhTris > 0)
    for (int k = 0; k < 3; k++)
      if (!(eye[k] >= ctx->bvhReach[k] && eye[k] <= ctx->bvhReach[3 + k])) ctx->sceneDirty = true;
  return RFX_OK;
}

// ----------------------------------------------------------------------------------------------------------- seeds
int rfx_set_seeds(rfx_ctx * ctx, uint32_t seed_vector3, uint32_t seed_render)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(ctx->dRng + ctx->rngSlot, &seed_vector3, sizeof(uint32_t), cudaMemcpyHostToDevice));
  ctx->seedRender = seed_render;
  return RFX_OK;
}

int rfx_get_seeds(rfx_ctx * ctx, uint32_t out[2])
{
  if (!ctx || !out) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(&out[0], ctx->dRng + ctx->rngSlot, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  out[1] = ctx->seedRender;
  return checkStatus(ctx);
}

int rfx_selftest_rng(rfx_ctx * ctx, uint64_t out[2])
{
  if (!ctx || !out) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  unsigned long long * d = nullptr;
  CK(cudaMalloc((void **)&d, 2 * sizeof(unsigned long long)));
  cudaError_t e = cudaMemset(d, 0, 2 * sizeof(unsigned long long));
  if (e == cudaSuccess) { ctx->stats.kernel_launches += launchRngSelftest(d, ctx->stream); e = cudaStreamSynchronize(ctx->stream); }
  unsigned long long h[2] = { 0, 0 };
  if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(ctx, RFX_ERR_CUDA, std::string("rfx_selftest_rng: ") + cudaGetErrorString(e));
  out[0] = h[0]; out[1] = h[1];
  return RFX_OK;
}

// The two host-side bound computations as pure functions (no device, no context), so that the CPU test suite can check them against
// the kernels' float32 expressions evaluated in numpy.
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
  FrameParams fp;
  memset(&fp, 0, sizeof(fp));
  memcpy(fp.eye, cam, 12); memcpy(fp.view, cam + 3, 36);
  fp.rz = float(width) / 2.0f / tanf(cam[12] / 2.0f);            // Render.cpp:148-150
  fp.wHalf = width / 2.0f; fp.hHalf = height / 2.0f;
  fp.W = width; fp.H = height;
  const PrimaryCull pc = makePrimaryCull(sc, fp);
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
  const double R = (double)reach_diagonal;
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
    const double noise = std::min(3e-7 * R * R / std::max((double)p.r, 1e-30), 7.7e-4 * R);   // as uploadScene sizes the box margins
    p.m = (float)(2.0 * noise + 1e-6 * R);
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
  FrameParams fp;
  memset(&fp, 0, sizeof(fp));
  memcpy(fp.eye, cam, 12); memcpy(fp.view, cam + 3, 36);
  fp.rz = float(width) / 2.0f / tanf(cam[12] / 2.0f);            // Render.cpp:148-150
  fp.wHalf = width / 2.0f; fp.hHalf = height / 2.0f;
  fp.W = width; fp.H = height;
  std::vector<float4> sp((size_t)n_spheres);
  for (int i = 0; i < n_spheres; i++) sp[i] = make_float4(spheres[4 * i], spheres[4 * i + 1], spheres[4 * i + 2], spheres[4 * i + 3]);
  int nx = 0, ny = 0;
  std::vector<uint32_t> cells;
  std::vector<float4> rec;
  std::vector<int> index;
  dims[0] = dims[1] = dims[2] = 0; counts[0] = counts[1] = 0;
  if (!binEyeGrid(fp, sp, nx, ny, cells, rec, index)) return RFX_OK;      // no grid for this camera: dims stay 0
  dims[0] = nx; dims[1] = ny; dims[2] = EYE_GRID_SHIFT;
  counts[0] = cells.size(); counts[1] = cells.back();
  if (cell_start && cell_cap >= cells.size()) memcpy(cell_start, cells.data(), cells.size() * sizeof(uint32_t));
  if (items && item_cap >= cells.back() && cells.back()) memcpy(items, index.data(), (size_t)cells.back() * sizeof(int32_t));
  return RFX_OK;
}

int rfx_selftest_primary_bounds(rfx_ctx * ctx, int32_t out[96], int32_t counts[2])
{
  if (!ctx || !out || !counts) return RFX_ERR_ARG;
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_primary_bounds: image size not set");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, ctx->stream)) != RFX_OK) return rc;
  if (!ctx->smallOk) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_primary_bounds: the scene does not fit the constant bank");
  FrameParams fp;
  memset(&fp, 0, sizeof(fp));
  memcpy(fp.eye, ctx->eye, sizeof(fp.eye));
  memcpy(fp.view, ctx->view, sizeof(fp.view));
  fp.rz = float(ctx->W) / 2.0f / tanf(ctx->fov / 2.0f);
  fp.wHalf = ctx->W / 2.0f;
  fp.hHalf = ctx->H / 2.0f;
  fp.W = ctx->W; fp.H = ctx->H;
  const PrimaryCull pc = makePrimaryCull(ctx->small, fp);
  static_assert(sizeof(pc.rect) == 96 * sizeof(int32_t), "24 rectangles of 4 ints");
  memcpy(out, pc.rect, sizeof(pc.rect));
  counts[0] = 0; counts[1] = ctx->small.nT;
  for (const HostObj & o : ctx->objs) counts[0] += o.kind == 0;      // (small.nS is padded to whole quads)
  return RFX_OK;
}

int rfx_skip_samples(rfx_ctx * ctx, uint64_t n)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  int rc;
  // the stream state lives on the device and advances in stream order: stay on the stream the renders use
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  const uint64_t chunk = 1ull << 28;
  while (n > 0)
  {
    const uint64_t m = std::min(n, chunk);
    if ((rc = rankSamples(ctx, m, true, st)) != RFX_OK) return rc;
    n -= m;
  }
  return RFX_OK;
}

// ---------------------------------------------------------------------------------------------------------- Render
int rfx_set_image_size(rfx_ctx * ctx, uint32_t width, uint32_t height)
{
  if (!ctx) return RFX_ERR_ARG;
  if (!width || !height) return fail(ctx, RFX_ERR_ARG, "rfx_set_image_size: zero size");   // Render.cpp:59-62: ignored
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  const size_t n = (size_t)width * height;
  if ((rc = ensure(ctx, ctx->dImage, ctx->imageCap, n * 3)) != RFX_OK) return rc;
  ctx->stats.kernel_launches += launchClear(ctx->dImage, n * 3, ctx->stream);   // Render.cpp:67-71
  CK(cudaGetLastError());
  ctx->W = width; ctx->H = height;
  ctx->additiveCounter = 0;
  ctx->inProgress = false;
  ctx->cursor = 0;
  return RFX_OK;
}

int rfx_render_begin(rfx_ctx * ctx, int reflect_num, int sample_num, int additive)
{
  if (!ctx) return RFX_ERR_ARG;
  if (reflect_num <= 0 || sample_num == 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_begin: reflect_num must be > 0 and sample_num != 0");
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_render_begin: image size not set");
  if (sample_num > 1024 || sample_num < -4096) return fail(ctx, RFX_ERR_ARG, "rfx_render_begin: sample_num out of range");
  ctx->reflNum = reflect_num;
  ctx->sampleNum = sample_num;
  ctx->additive = additive != 0;
  ctx->inProgress = true;
  ctx->cursor = 0;
  if (additive) ctx->additiveCounter++; else ctx->additiveCounter = 0;     // Render.cpp:130-133

  FrameParams & fp = ctx->snap;
  memset(&fp, 0, sizeof(fp));
  memcpy(fp.eye, ctx->eye, sizeof(fp.eye));      // renderCameraEye / renderCameraView snapshot, Render.cpp:125-126
  memcpy(fp.view, ctx->view, sizeof(fp.view));
  // Render.cpp:148-150.  NOTE the reference evaluates rz with the LIVE camera.fov inside renderNext; Pulse never changes
  // fov (Camera.cpp has no writer besides the constructors), so latching it here is equivalent.
  fp.rz = float(ctx->W) / 2.0f / tanf(ctx->fov / 2.0f);
  fp.wHalf = ctx->W / 2.0f;
  fp.hHalf = ctx->H / 2.0f;
  fp.W = ctx->W; fp.H = ctx->H;
  fp.reflNum = reflect_num;
  fp.sampleNum = sample_num;
  fp.jitter = additive ? 1 : 0;
  fp.accumulate = ctx->additiveCounter > 1 ? 1 : 0;
  return RFX_OK;
}

int rfx_render_next(rfx_ctx * ctx, uint32_t pixels)
{
  if (!ctx) return RFX_ERR_ARG;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!pixels || !ctx->inProgress || ctx->cursor >= total) return 0;     // Render.cpp:143-144: returns false
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, ctx->stream)) != RFX_OK) return rc;
  if (ctx->sigOn && (rc = ensure(ctx, ctx->dSig, ctx->sigCap, (size_t)total)) != RFX_OK) return rc;
  const uint64_t end = std::min(total, ctx->cursor + pixels);
  if ((rc = renderRange(ctx, ctx->cursor, end, nullptr, true, ctx->stream)) != RFX_OK) return rc;
  ctx->cursor = end;
  if (ctx->cursor >= total) ctx->inProgress = false;                     // Render.cpp:207-211
  return ctx->inProgress ? 1 : 0;
}

// number of Scene::trace calls the reference makes for pixels [p0, p1) of the latched frame
static uint64_t callsIn(const rfx_ctx * ctx, uint64_t p0, uint64_t p1)
{
  if (ctx->sampleNum > 0) return (p1 - p0) * (uint64_t)ctx->sampleNum * (uint64_t)ctx->sampleNum;
  const uint32_t a = (uint32_t)(-ctx->sampleNum);
  return originsBefore(p1, ctx->W, a) - originsBefore(p0, ctx->W, a);
}

static int skipPixels(rfx_ctx * ctx, uint64_t p0, uint64_t p1, cudaStream_t st)
{
  int rc;
  uint64_t n = callsIn(ctx, p0, p1);
  const uint64_t chunk = 1ull << 28;
  while (n > 0)
  {
    const uint64_t m = std::min(n, chunk);
    if ((rc = rankSamples(ctx, m, true, st)) != RFX_OK) return rc;
    n -= m;
  }
  if (ctx->snap.jitter && ctx->sampleNum > 0) ctx->seedRender = lcgJumpHost(ctx->seedRender, 2 * (p1 - p0));
  return RFX_OK;
}

int rfx_render_range(rfx_ctx * ctx, uint64_t p0, uint64_t p1, uint32_t * argb_device, void * stream)
{
  if (!ctx) return RFX_ERR_ARG;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!ctx->inProgress) return fail(ctx, RFX_ERR_ARG, "rfx_render_range: no frame in progress");
  if (p0 > p1 || p1 > total || p0 < ctx->cursor) return fail(ctx, RFX_ERR_ARG, "rfx_render_range: ranges must be increasing and inside the frame");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  if (ctx->sigOn && (rc = ensure(ctx, ctx->dSig, ctx->sigCap, (size_t)total)) != RFX_OK) return rc;
  if (p0 > ctx->cursor && (rc = skipPixels(ctx, ctx->cursor, p0, st)) != RFX_OK) return rc;
  if ((rc = renderRange(ctx, p0, p1, argb_device, argb_device == nullptr, st)) != RFX_OK) return rc;
  ctx->cursor = p1;
  return RFX_OK;
}

int rfx_render_strips(rfx_ctx * ctx, uint32_t strip_rows, uint32_t world, uint32_t rank, uint32_t * argb_device, void * stream)
{
  if (!ctx || !argb_device || !strip_rows || !world || rank >= world) return fail(ctx, RFX_ERR_ARG, "rfx_render_strips: bad argument");
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!ctx->inProgress || ctx->cursor != 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_strips: needs a freshly begun frame");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  const uint64_t calls = ctx->sampleNum > 0 ? callsIn(ctx, 0, total) : 0;
  const bool fast = ctx->sampleNum > 0 && ctx->smallOk && ctx->forcePath < 2 && !ctx->snap.jitter && !ctx->sigOn &&
                    strip_rows % 8 == 0 && calls <= (1ull << 26);
  if (!fast)
  {
    // general path: one range per strip (block preview, big scenes, huge SSAA factors)
    const uint32_t nStrips = (ctx->H + strip_rows - 1) / strip_rows;
    for (uint32_t s = rank; s < nStrips; s += world)
    {
      const uint64_t p0 = (uint64_t)s * strip_rows * ctx->W, p1 = std::min<uint64_t>(total, (uint64_t)(s + 1) * strip_rows * ctx->W);
      if ((rc = rfx_render_range(ctx, p0, p1, argb_device, stream)) != RFX_OK) return rc;
    }
    return rfx_render_finish(ctx);
  }
  const uint64_t perPixel = (uint64_t)ctx->sampleNum * ctx->sampleNum;
  // K1 once over the whole frame (every GPU needs the accept counts of everything before its rows); only the states of
  // this rank's strips are stored
  if ((rc = rankSamples(ctx, calls, false, st, (uint64_t)strip_rows * ctx->W * perPixel, world, rank)) != RFX_OK) return rc;
  TraceWork w;
  w.sceneBlob = ctx->dBlob; w.sceneBytes = ctx->blobBytes;
  w.fp = ctx->snap;
  w.fp.p0 = 0; w.fp.p1 = total; w.fp.firstRank = 0; w.fp.seedRender = ctx->seedRender;
  w.fp.stripRows = strip_rows; w.fp.stripWorld = world; w.fp.stripRank = rank;
  w.sampleStates = ctx->dSampleStates;
  w.image = nullptr; w.argbOut = argb_device; w.sigOut = nullptr; w.counters = ctx->dCounters;
  w.lightGrids = ctx->lightGridsBuilt > 0;
  w.triBvh = ctx->triBvhTris > 0;
  cudaEvent_t evA = nullptr, evB = nullptr;
  if (ctx->profiling)
  {
    if (ctx->evUsed + 2 > ctx->evPool.size())
      for (int i = 0; i < 2; i++) { cudaEvent_t e; CK(cudaEventCreate(&e)); ctx->evPool.push_back(e); }
    evA = ctx->evPool[ctx->evUsed++]; evB = ctx->evPool[ctx->evUsed++];
    CK(cudaEventRecord(evA, st));
  }
  if ((rc = armTileOrder(ctx, w, st)) != RFX_OK) return rc;
  {
    const int nl = launchTraceSmall(ctx->small, w, st);
    ctx->stats.kernel_launches += nl; ctx->stats.launches_small_fast += nl;
  }
  if (evB) CK(cudaEventRecord(evB, st));
  CK(cudaGetLastError());
  ctx->stats.samples += calls / world;
  ctx->cursor = total;
  ctx->inProgress = false;
  return RFX_OK;
}

int rfx_render_finish(rfx_ctx * ctx)
{
  if (!ctx) return RFX_ERR_ARG;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!ctx->inProgress) return RFX_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  int rc;
  if (ctx->cursor < total && (rc = skipPixels(ctx, ctx->cursor, total, st)) != RFX_OK) return rc;
  ctx->cursor = total;
  ctx->inProgress = false;
  return RFX_OK;
}

int rfx_buffer_alloc(rfx_ctx * ctx, uint64_t bytes, void ** device_ptr)
{
  if (!ctx || !device_ptr || !bytes) return fail(ctx, RFX_ERR_ARG, "rfx_buffer_alloc: bad argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMalloc(device_ptr, bytes));
  CK(cudaMemset(*device_ptr, 0, bytes));
  return RFX_OK;
}

int rfx_buffer_free(rfx_ctx * ctx, void * device_ptr)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaFree(device_ptr));
  return RFX_OK;
}

int rfx_buffer_read(rfx_ctx * ctx, const void * device_ptr, void * host_dst, uint64_t bytes)
{
  if (!ctx || !device_ptr || !host_dst) return fail(ctx, RFX_ERR_ARG, "rfx_buffer_read: NULL argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(host_dst, device_ptr, bytes, cudaMemcpyDeviceToHost));
  ctx->stats.d2h_bytes += bytes;
  return RFX_OK;
}

int rfx_ipc_export(rfx_ctx * ctx, void * device_ptr, unsigned char handle[64])
{
  if (!ctx || !device_ptr || !handle) return fail(ctx, RFX_ERR_ARG, "rfx_ipc_export: NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CK(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, device_ptr));
  memcpy(handle, &h, 64);
  return RFX_OK;
}

int rfx_ipc_import(rfx_ctx * ctx, const unsigned char handle[64], void ** device_ptr)
{
  if (!ctx || !device_ptr || !handle) return fail(ctx, RFX_ERR_ARG, "rfx_ipc_import: NULL argument");
  CK(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CK(cudaIpcOpenMemHandle(device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return RFX_OK;
}

int rfx_ipc_close(rfx_ctx * ctx, void * device_ptr)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaIpcCloseMemHandle(device_ptr));
  return RFX_OK;
}

float rfx_progress(const rfx_ctx * ctx)
{
  if (!ctx || !ctx->W || !ctx->H) return 0.0f;
  // float(curx + cury * imageWidth) * 100.0f / imageWidth / imageHeight, Render.cpp:223-226; a finished frame leaves the
  // cursor at (0, imageHeight) upstream, i.e. 100 %
  return float(ctx->cursor) * 100.0f / ctx->W / ctx->H;
}

int rfx_additive_counter(const rfx_ctx * ctx) { return ctx ? ctx->additiveCounter : 0; }
int rfx_in_progress(const rfx_ctx * ctx) { return ctx && ctx->inProgress ? 1 : 0; }

static int readResolved(rfx_ctx * ctx, float * rgbf, uint32_t * argb, int divide = 1)
{
  const int counter = divide ? ctx->additiveCounter : 0;
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "image size not set");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  const size_t n = (size_t)ctx->W * ctx->H;
  if (argb)
  {
    if ((rc = ensure(ctx, ctx->dResolve, ctx->resolveCap, n)) != RFX_OK) return rc;
    ctx->stats.kernel_launches += launchResolve(ctx->dImage, n, counter, nullptr, ctx->dResolve, ctx->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(argb, ctx->dResolve, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.d2h_bytes += n * 4;
  }
  if (rgbf)
  {
    if (counter > 1)
    {
      // divide on the device into the ranked-state scratch (reused as a float buffer), then copy
      size_t need = n * 3;
      if ((rc = ensure(ctx, ctx->dSampleStates, ctx->statesCap, need)) != RFX_OK) return rc;
      ctx->stats.kernel_launches += launchResolve(ctx->dImage, n, counter, reinterpret_cast<float *>(ctx->dSampleStates), nullptr, ctx->stream);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(rgbf, ctx->dSampleStates, n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    }
    else
      CK(cudaMemcpyAsync(rgbf, ctx->dImage, n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.d2h_bytes += n * 12;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return checkStatus(ctx);
}

int rfx_read_argb(rfx_ctx * ctx, uint32_t * dst)
{
  if (!ctx || !dst) return fail(ctx, RFX_ERR_ARG, "rfx_read_argb: NULL argument");
  return readResolved(ctx, nullptr, dst);
}

int rfx_read_rgbf(rfx_ctx * ctx, float * dst)
{
  if (!ctx || !dst) return fail(ctx, RFX_ERR_ARG, "rfx_read_rgbf: NULL argument");
  return readResolved(ctx, dst, nullptr);
}

int rfx_read_image(rfx_ctx * ctx, float * rgbf, uint32_t * argb, int divide)
{
  if (!ctx || (!rgbf && !argb)) return fail(ctx, RFX_ERR_ARG, "rfx_read_image: NULL argument");
  return readResolved(ctx, rgbf, argb, divide);
}

int rfx_trace_rays(rfx_ctx * ctx, int n, const float * origins, const float * rays, int reflect_num, float * rgb)
{
  if (!ctx || n < 0 || !origins || !rays || !rgb || reflect_num <= 0) return fail(ctx, RFX_ERR_ARG, "rfx_trace_rays: bad argument");
  if (n == 0) return RFX_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  if (ctx->bvhDepth > 0 || ctx->triBvhTris > 0)
  {
    // the hierarchies' box margins are sized for ray origins inside bvhReach: origins outside it widen the region and re-flatten
    bool outside = false;
    for (int i = 0; i < n; i++)
      for (int k = 0; k < 3; k++)
      {
        const float v = origins[3 * (size_t)i + k];
        if (!(v >= ctx->bvhReach[k] && v <= ctx->bvhReach[3 + k]) && v == v && fabsf(v) <= FLT_MAX)
        {
          outside = true;
          ctx->extraOrigins[k] = std::min(ctx->extraOrigins[k], v);
          ctx->extraOrigins[3 + k] = std::max(ctx->extraOrigins[3 + k], v);
        }
      }
    if (outside)
    {
      ctx->sceneDirty = true;
      if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
    }
  }
  if ((rc = rankSamples(ctx, (uint64_t)n, false, st)) != RFX_OK) return rc;
  // ray buffers: origins | rays | rgb in one scratch allocation
  if ((rc = ensure(ctx, ctx->dRays, ctx->raysCap, (size_t)n * 9)) != RFX_OK) return rc;
  float * dO = ctx->dRays, * dR = ctx->dRays + (size_t)n * 3, * dC = ctx->dRays + (size_t)n * 6;
  CK(cudaMemcpyAsync(dO, origins, (size_t)n * 12, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(dR, rays, (size_t)n * 12, cudaMemcpyHostToDevice, st));
  ctx->stats.h2d_bytes += (uint64_t)n * 24;
  ctx->stats.kernel_launches += launchTraceBlobRays(ctx->dBlob, n, dO, dR, reflect_num, ctx->dSampleStates, dC, ctx->dCounters, st, ctx->triBvhTris > 0);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(rgb, dC, (size_t)n * 12, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  ctx->stats.d2h_bytes += (uint64_t)n * 12;
  ctx->stats.samples += (uint64_t)n;
  return checkStatus(ctx);
}

int rfx_read_pixel(rfx_ctx * ctx, int x, int y, float rgb[3])
{
  if (!ctx || !rgb) return RFX_ERR_ARG;
  rgb[0] = rgb[1] = rgb[2] = 0.0f;                                        // Render.cpp:112-113
  if (x < 0 || y < 0 || (uint32_t)x >= ctx->W || (uint32_t)y >= ctx->H) return RFX_OK;
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  CK(cudaMemcpyAsync(rgb, ctx->dImage + ((size_t)y * ctx->W + x) * 3, 12, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->stats.d2h_bytes += 12;
  if (ctx->additiveCounter > 1)
  {
    const float d = float(ctx->additiveCounter);                         // Render.cpp:109-110, Color.cpp:99-107
    rgb[0] = rgb[0] / d; rgb[1] = rgb[1] / d; rgb[2] = rgb[2] / d;
  }
  return RFX_OK;
}

int rfx_enable_signatures(rfx_ctx * ctx, int on)
{
  if (!ctx) return RFX_ERR_ARG;
  ctx->sigOn = on != 0;
  return RFX_OK;
}

int rfx_read_signatures(rfx_ctx * ctx, uint32_t * dst)
{
  if (!ctx || !dst) return RFX_ERR_ARG;
  if (!ctx->sigOn || !ctx->dSig) return fail(ctx, RFX_ERR_ARG, "rfx_read_signatures: signatures are not enabled");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  CK(cudaMemcpyAsync(dst, ctx->dSig, (size_t)ctx->W * ctx->H * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return RFX_OK;
}

// ----------------------------------------------------------------------------------------------------- batch path
static int beginFrame(rfx_ctx * ctx, const float * cam, int reflect_num, int sample_num)
{
  int rc;
  if ((rc = rfx_set_camera(ctx, cam, cam + 3, cam[12])) != RFX_OK) return rc;
  ctx->additiveCounter = 0;   // each frame is a fresh setImageSize-sized, non-additive screenshot render (Pulse.cpp:174-176)
  return rfx_render_begin(ctx, reflect_num, sample_num, 0);
}

int rfx_render_frames_device(rfx_ctx * ctx, int n_frames, const float * cams, int reflect_num, int sample_num,
                             uint32_t * argb_device, void * stream)
{
  if (!ctx || !cams || !argb_device || n_frames < 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames_device: bad argument");
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames_device: image size not set");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  // one K1 pass ranks the random states of a whole group of frames (the stream simply continues from frame to frame)
  if (reflect_num <= 0 || sample_num == 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames_device: reflect_num must be > 0 and sample_num != 0");
  ctx->sampleNum = sample_num;
  const uint64_t perFrame = callsIn(ctx, 0, total);
  const int group = (int)std::max<uint64_t>(1, ctx->maxCallsPerLaunch / std::max<uint64_t>(perFrame, 1));
  for (int f0 = 0; f0 < n_frames; f0 += group)
  {
    const int g = std::min(group, n_frames - f0);
    const bool pre = perFrame <= ctx->maxCallsPerLaunch;
    if (pre && (rc = rankSamples(ctx, perFrame * g, false, st)) != RFX_OK) return rc;
    for (int f = f0; f < f0 + g; f++)
    {
      if ((rc = beginFrame(ctx, cams + 13 * (size_t)f, reflect_num, sample_num)) != RFX_OK) return rc;
      if (ctx->sceneDirty && (rc = uploadScene(ctx, st)) != RFX_OK) return rc;   // this frame's eye left the box the BVH margins were sized for
      if ((rc = renderRange(ctx, 0, total, argb_device + (size_t)f * total, false, st,
                            pre ? ctx->dSampleStates + (size_t)(f - f0) * perFrame : nullptr)) != RFX_OK) return rc;
      ctx->cursor = total;
      ctx->inProgress = false;
    }
  }
  return RFX_OK;
}

int rfx_render_frames(rfx_ctx * ctx, int n_frames, const float * cams, int reflect_num, int sample_num, uint32_t * argb_host)
{
  if (!ctx || !cams || !argb_host || n_frames < 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames: bad argument");
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames: image size not set");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  // FRAME_SLOTS device frame slots: render frame f into slot f % FRAME_SLOTS on the compute stream while the copy stream(s)
  // drain older slots into the caller's host buffer
  const int NS = rfx_ctx::FRAME_SLOTS;
  if (ctx->frameCap < total || !ctx->dFrame[0])
  {
    CK(cudaDeviceSynchronize());
    for (int j = 0; j < NS; j++) { if (ctx->dFrame[j]) cudaFree(ctx->dFrame[j]); ctx->dFrame[j] = nullptr; }
    ctx->frameCap = 0;
    for (int j = 0; j < NS; j++) CK(cudaMalloc((void **)&ctx->dFrame[j], total * 4));
    ctx->frameCap = total;
  }
  if (reflect_num <= 0 || sample_num == 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames: reflect_num must be > 0 and sample_num != 0");
  ctx->sampleNum = sample_num;
  const uint64_t perFrame = callsIn(ctx, 0, total);
  const int group = (int)std::max<uint64_t>(1, ctx->maxCallsPerLaunch / std::max<uint64_t>(perFrame, 1));
  const bool pre = perFrame <= ctx->maxCallsPerLaunch;
  for (int f = 0; f < n_frames; f++)
  {
    const int slot = f % NS;
    cudaStream_t cs = ctx->copyStream[ctx->copyStreams > 1 ? (f & 1) : 0];
    if (pre && f % group == 0 && (rc = rankSamples(ctx, perFrame * std::min(group, n_frames - f), false, st)) != RFX_OK) return rc;
    if (f >= NS) CK(cudaStreamWaitEvent(st, ctx->evCopied[slot], 0));   // slot free again?
    if ((rc = beginFrame(ctx, cams + 13 * (size_t)f, reflect_num, sample_num)) != RFX_OK) return rc;
    if (ctx->sceneDirty && (rc = uploadScene(ctx, st)) != RFX_OK) return rc;   // this frame's eye left the box the BVH margins were sized for
    if ((rc = renderRange(ctx, 0, total, ctx->dFrame[slot], false, st,
                          pre ? ctx->dSampleStates + (size_t)(f % group) * perFrame : nullptr)) != RFX_OK) return rc;
    ctx->cursor = total;
    ctx->inProgress = false;
    CK(cudaEventRecord(ctx->evRendered[slot], st));
    CK(cudaStreamWaitEvent(cs, ctx->evRendered[slot], 0));
    CK(cudaMemcpyAsync(argb_host + (size_t)f * total, ctx->dFrame[slot], total * 4, cudaMemcpyDeviceToHost, cs));
    CK(cudaEventRecord(ctx->evCopied[slot], cs));
    ctx->stats.d2h_bytes += total * 4;
  }
  for (int i = 0; i < 2; i++) CK(cudaStreamSynchronize(ctx->copyStream[i]));
  CK(cudaStreamSynchronize(st));
  return checkStatus(ctx);
}

int rfx_synchronize(rfx_ctx * ctx)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  if (ctx->lastStream) CK(cudaStreamSynchronize(ctx->lastStream));
  CK(cudaStreamSynchronize(ctx->stream));
  return checkStatus(ctx);
}

// ----------------------------------------------------------------------------------------------------------- stats
int rfx_get_stats(rfx_ctx * ctx, rfx_stats * out)
{
  if (!ctx || !out) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  unsigned long long c[64];
  CK(cudaMemcpy(c, ctx->dCounters, sizeof(c), cudaMemcpyDeviceToHost));
  uint64_t b = 0, s = 0;
  for (int i = 0; i < 32; i++) { b += c[2 * i]; s += c[2 * i + 1]; }
  ctx->stats.bounces = b;
  ctx->stats.shadow_rays = s;
  ctx->stats.rays = b + s;
  for (size_t i = 0; i + 1 < ctx->evUsed; i += 2)
  {
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->evPool[i], ctx->evPool[i + 1]));
    ctx->stats.trace_kernel_ms += ms;
    ctx->stats.trace_kernels++;
  }
  ctx->evUsed = 0;
  ctx->stats.light_grids = (uint64_t)ctx->lightGridsBuilt;
  ctx->stats.bvh_triangles = ctx->triBvhTris;
  *out = ctx->stats;
  return RFX_OK;
}

int rfx_stats_reset(rfx_ctx * ctx)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemset(ctx->dCounters, 0, 64 * sizeof(unsigned long long)));
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->evUsed = 0;
  return RFX_OK;
}

int rfx_force_path(rfx_ctx * ctx, int path)
{
  if (!ctx || path < 0 || path > 3) return RFX_ERR_ARG;
  ctx->forcePath = path;
  return RFX_OK;
}

int rfx_set_tile_ordering(rfx_ctx * ctx, int on)
{
  if (!ctx) return RFX_ERR_ARG;
  ctx->tileOrdering = on != 0;
  ctx->tileHistory = false;
  return RFX_OK;
}

int rfx_set_bvh_mode(rfx_ctx * ctx, int mode)
{
  if (!ctx || mode < 0 || mode > 2) return RFX_ERR_ARG;
  ctx->bvhMode = mode;
  ctx->sceneDirty = true;
  return RFX_OK;
}

int rfx_set_option(rfx_ctx * ctx, const char * name, int64_t value)
{
  if (!ctx || !name) return RFX_ERR_ARG;
  if (!strcmp(name, "max_calls_per_launch"))
  {
    if (value < 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: max_calls_per_launch must be >= 1");
    ctx->maxCallsPerLaunch = (uint64_t)value;
    return RFX_OK;
  }
  if (!strcmp(name, "light_grids"))
  {
    if (value != 0 && value != 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: light_grids must be 0 or 1");
    if (ctx->lightGridsOn != (value != 0)) ctx->sceneDirty = true;
    ctx->lightGridsOn = value != 0;
    return RFX_OK;
  }
  if (!strcmp(name, "eye_grid"))
  {
    if (value != 0 && value != 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: eye_grid must be 0 or 1");
    ctx->eyeGridOn = value != 0;
    ctx->eyeValid = false;
    return RFX_OK;
  }
  if (!strcmp(name, "blob_wavefront"))
  {
    if (value < 0 || value > 64) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: blob_wavefront must be 0 (off) or the number of first segments (1..64)");
    ctx->blobWavefront = (int)value;
    return RFX_OK;
  }
  if (!strcmp(name, "tile_order_period"))
  {
    if (value < 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: tile_order_period must be >= 1");
    ctx->tileRecordPeriod = (int)std::min<int64_t>(value, 1 << 30);
    return RFX_OK;
  }
  if (!strcmp(name, "blob_smem_bvh"))
  {
    ctx->blobSmemBvh = value != 0;
    return RFX_OK;
  }
  if (!strcmp(name, "copy_streams"))
  {
    if (value < 1 || value > 2) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: copy_streams must be 1 or 2");
    ctx->copyStreams = (int)value;
    return RFX_OK;
  }
  return fail(ctx, RFX_ERR_ARG, std::string("rfx_set_option: unknown option ") + name);
}

int rfx_enable_profiling(rfx_ctx * ctx, int on)
{
  if (!ctx) return RFX_ERR_ARG;
  ctx->profiling = on != 0;
  return RFX_OK;
}

} // extern "C"
