// rfx_types.h — POD records shared by the host flattening code (rfx_scene.cpp) and the sm_100a kernels (rfx_kernels.cu).
//
// HBM layout of a scene ("scene blob", one contiguous allocation, read in place by k_trace):
//   SceneHeader | Light[nLights] | float4 sphere[nSpheres] (cx,cy,cz,r^2) | Triangle[nTris] | Plane[nPlanes] |
//   Material[nObjects] (sorted order: spheres, triangles, planes) | TexRef[nTextures]
// Objects are grouped by kind so the intersection loops are branch-free over a homogeneous array; every record keeps
// the object's insertion index so closest-hit ties resolve exactly as the reference's list walk does
// (first inserted wins, reference Scene.cpp:98) and the shadow loop can skip the hit object (Scene.cpp:135).
#pragma once
#include <stdint.h>
#include <vector_types.h>

namespace rfx
{

struct Material          // reference Material.h:8-12 (+ where the colour comes from)
{
  float r, g, b;
  float reflectivity;
  int type;              // 0 metal, 1 dielectric
  int order;             // insertion index in the reference's sceneObjects list
  int tex;               // triangles: texture id or -1
  int pad;
};

struct Light             // reference OmniLight.h:8-11
{
  float ox, oy, oz, radius;
  float r, g, b, power;
};

struct Triangle          // reference Triangle.h:10-16 (what trace() reads)
{
  float v0[3];
  float ax[9];           // axTrans = inverse[ v2-v0 | v1-v0 | -n ], row-major
  float n[3];
  float tuv[4];          // tuvTrans rows 1-2, columns 1-2 (column 3 and row 3 only ever meet zeros)
  float tu0, tv0;
};

struct Plane             // reference Plane.h
{
  float pos[3];
  float n[3];
};

struct TexRef
{
  const uint32_t * px;   // device pointer, 0xAARRGGBB, row 0 = v 0; NULL = empty texture (checker fallback)
  uint32_t w, h;
};

// Shadow-ray candidates of one far light (built by rfx_scene.cpp next to the hierarchy, walked by rfx_trace_blob.cu).  Every shadow ray
// towards the light is nearly parallel to the direction from the scene to the light, so the spheres it can hit are the ones whose
// (inflated) shadow on a plane across that direction covers the ray's origin: a 2-D grid of candidate lists over that plane.
struct LightGrid
{
  float u[4], v[4];                 // cell of a point p: column floor(u[0] p.x + u[1] p.y + u[2] p.z + u[3]), row likewise with v
  int nx, ny;
  const uint32_t * cellStart;       // [nx * ny + 1] offsets into the item arrays; NULL: no grid for this light (queries walk the hierarchy)
  const float4 * itemSphere;        // candidate spheres (cx, cy, cz, r^2), cell after cell
  const int * itemIndex;            // their positions in the sorted sphere array (materials, tie-break order, the skipped object)
};

struct SceneHeader
{
  int nSpheres, nTris, nPlanes, nLights, nTextures;
  int skyTex;                       // texture id or -1
  float ambient[3], ambientPower;   // Scene::diffLightColor / diffLightPower
  float env[3];                     // Scene::envColor
  float halfTileW, halfTileH;       // Skybox::halfTileWidth/Height
  uint32_t offLights, offSpheres, offTris, offPlanes, offMats, offTex;   // byte offsets inside the blob
  uint32_t bytes;                   // blob size
  const float * byteLut;            // 256 floats: float(i) / 255.0f computed on the host (reference Color.cpp:11-13)
  const int * bvhPrims;             // big scenes: sphere indices (sorted-array positions) of the leaf slots, 4 slots per leaf (-1 = unused)
  const float4 * bvhPairs;          // NULL: no hierarchy (list walk).  Inner nodes with both children's boxes: 4 float4 per node {lo_a, ref_a} {hi_a, ref_b} {lo_b, -} {hi_b, -}; ref >= 0 pair node, < 0 ~leaf slot
  int bvhRoot;                      // ref of the root (a pair node, or a leaf when there are <= 4 spheres)
  const float4 * bvhLeafSph;        // the same slots as (cx, cy, cz, r^2), NaN = unused: a leaf is 4 contiguous records
  uint32_t bvhFloat4;               // float4 count of [leaf records | pair nodes], contiguous from bvhLeafSph (what a CTA copies to shared memory)
  const LightGrid * lightGrids;     // [nLights] when the hierarchy exists and some light is far enough for a grid, else NULL
  // hierarchy over the triangles (rfx_scene.cpp buildTriBoxes), walked after the spheres; triPairs == NULL: list walk.  Same pair-node
  // format and leaf refs as the sphere hierarchy; a leaf slot is 3 float4 {v0.xyz, ax6} {ax7, ax8, ax0, ax1} {ax2, ax3, ax4, ax5}
  // (as SmallScene::triPk), all zero in unused slots (ax row 3 = 0: |rz| > 2^-63 never holds)
  const int * triPrims;             // position in the sorted triangle array of each leaf slot, 4 slots per leaf (-1 = unused)
  const float4 * triLeaf;           // 3 float4 per slot, then the pair nodes
  const float4 * triPairs;
  int triRoot;
  // Scenes with a plane and a hierarchy (rfx_scene.cpp farGrowthSpheres): a drop point on a plane can lie outside the box of ray origins
  // the margins were sized for.  A query whose origin o lies outside a reach box grows every box of that hierarchy by
  // grow * (L1 distance of o from the reach box); from inside it grows nothing.  Only the kernels instantiated with FAR read these.
  float sphReach[6];                // lo xyz, hi xyz: the box the sphere margins assume (every origin and every centre)
  float triReach[6];                // the same for the triangle margins (sphReach joined with every effective triangle)
  float growS, growT;               // growth per unit of distance, rounded upwards
  const int * triAlways;            // plane scenes: triangles no margin can hold from far origins (slivers, non-finite), sorted-array
  int nTriAlways;                   // positions, tested one by one after the triangle walk; they are not in the hierarchy
};

// Small scenes travel as a kernel parameter (constant bank): see rfx_trace_small.cu
constexpr int SMALL_MAX_SPHERES = 16;
constexpr int SMALL_MAX_TRIS = 8;
constexpr int SMALL_MAX_PLANES = 2;
constexpr int SMALL_MAX_LIGHTS = 4;
constexpr int SMALL_MAX_TEX = 8;
constexpr int SMALL_MAX_OBJECTS = SMALL_MAX_SPHERES + SMALL_MAX_TRIS + SMALL_MAX_PLANES;

struct SmallScene
{
  int nS, nT, nP, nL;                       // nS: spheres padded to whole quads with NaN records (never hit)
  int skyTex;
  float halfTileW, halfTileH;
  float ambientPower;
  float ambient[3];
  float env[3];
  const float * byteLut;
  float4 sph[SMALL_MAX_SPHERES];            // cx, cy, cz, r^2
  Triangle tri[SMALL_MAX_TRIS];
  // the same triangles repacked for 64-bit constant loads in the intersection loop:
  // [0] = v0.x v0.y v0.z ax[6]   [1] = ax[7] ax[8] ax[0] ax[1]   [2] = ax[2] ax[3] ax[4] ax[5]
  float4 triPk[SMALL_MAX_TRIS][3];
  Plane pl[SMALL_MAX_PLANES];
  Light light[SMALL_MAX_LIGHTS];
  Material mat[SMALL_MAX_OBJECTS];          // indexed by candidate-mask bit: spheres 0.., triangles 16.., planes 24..
  TexRef tex[SMALL_MAX_TEX];
};

struct FrameParams                  // one renderBegin snapshot + the renderNext slice being rendered
{
  float eye[3];
  float view[9];                    // row-major _11.._33
  float rz, wHalf, hHalf;           // Render.cpp:148-150 (rz from host tanf)
  uint32_t W, H;
  int reflNum;                      // renderReflectNum
  int sampleNum;                    // renderSampleNum (> 0 grid SSAA, < 0 block preview)
  int jitter;                       // renderAdditive: draw rndx, rndy per pixel from the Render.cpp TU stream
  int accumulate;                   // additiveCounter > 1: image += colour
  uint32_t seedRender;              // Render.cpp TU LCG state at the first pixel of this slice
  uint64_t p0, p1;                  // linear pixel range [p0, p1) of this slice, scan order (y-major)
  uint64_t firstRank;               // block-preview mode: number of block origins before p0
  uint32_t stripRows, stripWorld, stripRank;   // split-frame mode (stripWorld > 0): this launch owns strips s with s % stripWorld == stripRank
};

struct Counters                     // device-side event counters (uint64 each)
{
  unsigned long long rays, bounces, shadowRays, samples;
};

} // namespace rfx
