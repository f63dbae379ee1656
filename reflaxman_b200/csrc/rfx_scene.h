// rfx_scene.h — host-side scene flattening: the host scene the C ABI collects, and the scene image built from it (blob, hierarchies,
// light grids, constant-bank form) that rfx_capi.cu uploads.  Pure host code: rfx_scene.cpp makes no CUDA runtime call.
//
// Host-side float arithmetic here (triangle basis inversion, skybox half-tile, rz) restates what the reference's constructors compute
// once per object/frame; it is compiled with -ffp-contract=off so every operation is the same IEEE binary32 operation the reference's
// build performs (reference Triangle.cpp:11-21,110-120; Matrix33.cpp:10-15,49-79; Skybox.cpp:21-37; Material.cpp:8-14; Render.cpp:148-150).
#pragma once
#include "rfx_types.h"

#include <float.h>
#include <math.h>
#include <string>
#include <vector>

namespace rfx
{

const float VSN = 1.08420217248550443e-19f;   // sqrtf(FLT_MIN), reference trace_math.h:17

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
void invertColumns(H3 u, H3 v, H3 n, float out[9]);
Material makeMaterial(int mtype, const float rgb[3], float refl, float transp, int order);   // Material.cpp:8-14

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

struct HostScene
{
  float ambient[3] = { 0, 0, 0 }, ambientPower = 0, env[3] = { 0, 0, 0 };
  std::vector<Light> lights;
  std::vector<HostObj> objs;
  std::vector<HostTex> tex;                 // uploaded before the image is built: TexRef and SmallScene carry their device pointers
  int skyTex = -1;
  int bvhMode = 0;                          // 0 auto (spheres > 32, triangles > 32), 1 always, 2 never (no plane: 0, 1) — tests compare them
  bool lightGridsOn = true;                 // rfx_set_option "light_grids"
  // ray origins the hierarchies' box margins must cover (besides every drop point)
  float eye[3] = { 0, 0, 0 };               // the camera's
  float extraOrigins[6] = { FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX };   // box of the ray origins rfx_trace_rays was given
};

// Device form of a hierarchy: leaf slots (4 per leaf, in node order), then the pair nodes (rfx_types.h SceneHeader)
struct PackedBvh
{
  std::vector<float4> nodes;                // empty: no hierarchy
  std::vector<int> prims;                   // per leaf slot: position in the sorted primitive array (-1 unused)
  int root = 0;                             // ref of the root
  size_t leafFloat4 = 0;                    // float4s of the leaf slots: the pair nodes start there
};

// Everything the device scene is made of.  Device pointers are left null — the blob header's byteLut, hierarchy and grid pointers,
// the light grids' arrays, SmallScene::byteLut — for the uploader to fill in once the arrays have their addresses.
struct SceneImage
{
  std::vector<unsigned char> blob;          // the blob layout of rfx_types.h, SceneHeader first
  std::vector<float4> spheres;              // the sorted sphere array (cx, cy, cz, r^2), as in the blob
  PackedBvh sphBvh, triBvh;
  // shadow-ray candidate grids of the far lights (LightGrid): empty when no light has one; grids[i].nx == 0: none for light i
  std::vector<LightGrid> grids;
  std::vector<uint32_t> gridCells;          // every grid's cell offsets, light after light (relative to the light's own items)
  std::vector<float4> gridSpheres;          // every grid's items, light after light
  std::vector<int> gridIndex;
  std::vector<size_t> gridCellOff, gridItemOff;   // per light: where its cells / items start in the arrays above
  int lightGridsBuilt = 0;
  SmallScene small;                         // constant-bank form of the same scene (rfx_trace_small.cu), when smallOk
  bool smallOk = false;
  float reach[6] = { 0, 0, 0, 0, 0, 0 };   // box of ray origins the hierarchies' margins were sized for (lo xyz, hi xyz)
  int bvhDepth = 0;                         // depth of the sphere hierarchy (0: none)
  uint32_t bvhFloat4 = 0;                   // SceneHeader::bvhFloat4
  uint64_t triBvhTris = 0;                  // triangles under the triangle hierarchy (0: list walk)
};

// flattens the host scene into img, rebuilt in place: its arrays keep their memory from the last image (a re-flatten of a big scene then
// touches no fresh pages).  RFX_ERR_ARG (with err, img unchanged) when the blob outgrows its 32-bit offsets.
int buildSceneImage(const HostScene & s, SceneImage & img, std::string & err);

// camera fields of a frame (the rest zero)
FrameParams frameFromCamera(const float eye[3], const float view[9], float fov, uint32_t W, uint32_t H);

// candidates of the first query of a path (EyeGrid, rfx_kernels.h): the primary-ray screen bounds of spheres[i] = (cx, cy, cz, r^2)
// binned into 2^EYE_GRID_SHIFT-pixel square cells; false: no grid for this camera
constexpr int EYE_GRID_SHIFT = 5;      // 32x32-pixel cells: a 4x8 tile of the kernels lies in one cell
bool binEyeGrid(const FrameParams & fp, const std::vector<float4> & spheres, int & nx, int & ny, std::vector<uint32_t> & cells,
                std::vector<float4> & items, std::vector<int> & index);

} // namespace rfx
