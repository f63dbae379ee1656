// rfx_scene.h — host-side scene flattening: the host scene the C ABI collects, and the scene image built from it (blob, hierarchies,
// light grids, constant-bank form) that rfx_capi.cu uploads.  Pure host code: rfx_scene.cpp makes no CUDA runtime call.
//
// Host-side float arithmetic here (triangle basis inversion, skybox half-tile, rz) restates what the reference's constructors compute
// once per object/frame; it is compiled with -ffp-contract=off so every operation is the same IEEE binary32 operation the reference's
// build performs (reference Triangle.cpp:11-21,110-120; Matrix33.cpp:10-15,49-79; Skybox.cpp:21-37; Material.cpp:8-14; Render.cpp:148-150).
#pragma once
#include "rfx_light_grid.h"

#include <float.h>
#include <math.h>
#include <string>
#include <vector>

namespace rfx
{

inline float clampf(float v, float lo, float hi) { return v < lo ? lo : v > hi ? hi : v; }

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

// A mesh of rfx_add_mesh: its triangles are objs[first, first + idx.size() / 3).  rfx_update_mesh replaces xyz and marks it stale:
// the triangles' host records (triVerts, tri) are recomputed from xyz before the next flatten (refreshMeshes).
struct HostMesh
{
  int first = 0;
  std::vector<uint32_t> idx;                // 3 per triangle
  std::vector<float> xyz;                   // the current vertices, 3 per vertex
  float box[6];                             // their box (lo xyz, hi xyz)
  bool stale = false;
};

struct HostScene
{
  float ambient[3] = { 0, 0, 0 }, ambientPower = 0, env[3] = { 0, 0, 0 };
  std::vector<Light> lights;
  std::vector<float> lightPower;            // per light: its power as given (the record keeps it clamped; env adds it unclamped, Scene.cpp:54)
  std::vector<HostObj> objs;
  std::vector<HostMesh> meshes;
  std::vector<HostTex> tex;                 // uploaded before the image is built: TexRef and SmallScene carry their device pointers
  int skyTex = -1;
  int bvhMode = 0;                          // 0 auto (spheres > 32, triangles > 32), 1 always, 2 never — tests compare them
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
  int lightGridsBuilt = 0;                  // lights the flatten built a grid for.  Not changed by later updates: > 0 means the device has a
                                            // header per light and grid regions, and gridBox, dropTris, dropSpheres stay tracked
  SmallScene small;                         // constant-bank form of the same scene (rfx_trace_small.cu), when smallOk
  bool smallOk = false;
  float reach[6] = { 0, 0, 0, 0, 0, 0 };   // box of ray origins the hierarchies' margins were sized for (lo xyz, hi xyz)
  int bvhDepth = 0;                         // depth of the sphere hierarchy (0: none)
  uint32_t bvhFloat4 = 0;                   // SceneHeader::bvhFloat4
  uint64_t triBvhTris = 0;                  // triangles under the triangle hierarchy (0: list walk)
  uint64_t bvhSpheres = 0;                  // spheres under the sphere hierarchy (0: list walk)
  std::vector<int> triAlways;               // SceneHeader::triAlways (plane scenes: triangles tested after the walk)
  bool far = false;                         // the scene has a plane and a hierarchy: the kernels instantiated with FAR
  // What rfx_update_mesh needs to set up mesh triangles and refit the triangle hierarchy on the device (rfx_mesh.cu) without a
  // re-flatten.  meshes[i] is scene.meshes[i] as flattened: its triangles sit at [triBase, triBase + nTris) of the sorted triangle
  // array, its index list at meshIdx[idxOff ...].
  struct MeshImage { int triBase; uint32_t nTris; size_t idxOff; };
  std::vector<MeshImage> meshes;
  std::vector<uint32_t> meshIdx;
  std::vector<int> triSlot;                 // per triangle of the sorted array: its leaf slot in triBvh, -1 (none); empty: no hierarchy
  std::vector<int> leafParent, pairParent;  // triBvh: per leaf / pair node, 2 * (parent pair node) + side (0: a, 1: b); -1: the root
  double triUnion[6] = { 0, 0, 0, 0, 0, 0 };  // the box R is the diagonal of in the triangle margins: reach joined with every E
  double gridBox[6] = { 0, 0, 0, 0, 0, 0 };   // the padded drop-point box the light grids were built for (when lightGridsBuilt)
  // The un-padded drop-point boxes (when lightGridsBuilt) that, joined with the meshes' current boxes, must stay inside gridBox for the
  // light grids to stay complete: the triangles outside meshes (fixed until the next flatten), and every sphere (rfx_update_spheres
  // keeps it current).  Empty: lo > hi.
  double dropTris[6] = { 0, 0, 0, 0, 0, 0 };
  double dropSpheres[6] = { 0, 0, 0, 0, 0, 0 };
  // What rfx_update_spheres needs to move spheres on the device (rfx_mesh.cu) without a re-flatten.  Spheres keep insertion order in
  // the sorted array: sphObj[i] is the object index of sphere i (ascending).
  std::vector<int> sphObj;
  std::vector<float> sphRadius;             // per sphere: its radius (the margins of the sphere hierarchy)
  std::vector<int> sphSlot;                 // per sphere: its leaf slot in sphBvh (the inverse of sphBvh.prims); empty: no hierarchy
  std::vector<int> sphLeafParent, sphPairParent;   // sphBvh, as leafParent / pairParent (blob scenes with a sphere hierarchy)
  double sphR = 0.0;                        // R of the sphere margins (the diagonal of reach)
};

// the drop-point box (lo xyz, hi xyz) padded for the rounding of a drop point, as the light grids take it
void padDropBox(double b[6]);

// the un-padded drop-point box (lo xyz, hi xyz) of the spheres of img, from their records in s
void sphereDropBox(const HostScene & s, const SceneImage & img, double b[6]);

// Builds into out's grid fields (grids, gridCells, gridSpheres, gridIndex, their offsets, lightGridsBuilt) the light grids of the
// current lights and spheres of s over the drop-point box img's were built for (img.gridBox), with the margins of img's flatten
// (img.sphR) and its prims in slot order, as buildSceneImage would build them for that box: the host reference of the grids
// rfx_update_spheres and rfx_update_lights build on the device (rfx_selftest_light_grids).  The device pointers are left null.
void rebuildLightGrids(const HostScene & s, const SceneImage & img, SceneImage & out);

// recompute the host records (triVerts, tri.v0/ax/n) of the stale meshes' triangles from their current vertices
void refreshMeshes(HostScene & s);

// flattens the host scene into img, rebuilt in place: its arrays keep their memory from the last image (a re-flatten of a big scene then
// touches no fresh pages).  RFX_ERR_ARG (with err, img unchanged) when the blob outgrows its 32-bit offsets.
int buildSceneImage(const HostScene & s, SceneImage & img, std::string & err);

// camera fields of a frame (the rest zero)
FrameParams frameFromCamera(const float eye[3], const float view[9], float fov, uint32_t W, uint32_t H);

// candidates of the first query of a path (EyeGrid, rfx_kernels.h): the primary-ray screen bounds of spheres[i] = (cx, cy, cz, r^2)
// binned into 2^EYE_GRID_SHIFT-pixel square cells; false: no grid for this camera
bool binEyeGrid(const FrameParams & fp, const std::vector<float4> & spheres, int & nx, int & ny, std::vector<uint32_t> & cells,
                std::vector<float4> & items, std::vector<int> & index);

} // namespace rfx
