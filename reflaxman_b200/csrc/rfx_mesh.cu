// rfx_mesh.cu — rfx_update_mesh on the device: set up a mesh's triangles from new vertices (k_mesh_setup) and refit the triangle
// hierarchy over the new boxes (k_tri_refit), without a host re-flatten.  rfx_update_spheres likewise: write the moved spheres' records
// (k_sphere_scatter) and refit the sphere hierarchy (k_sphere_refit).
//
// Both kernels run the host's own per-triangle code (rfx_tri_setup.h: the reference's constructor, the box arithmetic of
// buildTriBoxes), compiled with --fmad=false, so every triangle record and every box is the one a host flatten of the same triangles
// would compute for the same R.  The hierarchy keeps the topology of the last flatten; only its boxes change.  R, the diagonal of the
// union of the reach box and every effective triangle, is taken over the union at the last flatten joined with the mesh's new
// effective triangles: it only grows until the next flatten, which keeps every margin sufficient.  A union box is an exact min / max,
// so a refit with unchanged vertices reproduces the host's packed hierarchy bit for bit.
#include "rfx_kernels.h"
#include "rfx_sphere_box.h"

namespace rfx
{

namespace
{

constexpr int SETUP_THREADS = 256;
constexpr int REFIT_THREADS = 128;

// The climb of a bottom-up refit, from a leaf whose box is (lo, hi) and whose parent ref is p (2 * pair node + side, -1: root): the
// thread writes its box into its side of the parent pair node (xyz lanes only: the w lanes hold the child refs); the second thread to
// arrive at a pair node unions its two children's boxes and carries on.  Returns true in the one thread that completed the root.
__device__ __forceinline__ bool refitClimb(float lo[3], float hi[3], int p, float4 * pairs, const int * pairParent, uint32_t * arrive)
{
  while (p >= 0)
  {
    const int node = p >> 1, side = p & 1;
    float * mine = reinterpret_cast<float *>(pairs + 4 * (size_t)node + 2 * side);   // {lo.xyz, ref} {hi.xyz, ref}
    mine[0] = lo[0]; mine[1] = lo[1]; mine[2] = lo[2];
    mine[4] = hi[0]; mine[5] = hi[1]; mine[6] = hi[2];
    __threadfence();
    if (atomicAdd(arrive + node, 1u) == 0) return false;   // the sibling's thread finishes this node
    __threadfence();
    const volatile float * other = reinterpret_cast<const volatile float *>(pairs + 4 * (size_t)node + 2 * (side ^ 1));
    for (int k = 0; k < 3; k++)
    {
      const float ol = other[k], oh = other[4 + k];
      lo[k] = ol < lo[k] ? ol : lo[k];
      hi[k] = hi[k] < oh ? oh : hi[k];
    }
    p = pairParent[node];
  }
  return true;
}

// One thread per mesh triangle: the triangle record in the blob (v0, ax, n; the texture fields stay), its leaf slot (packTriangle
// layout), and the block's union of the new effective triangles, folded into u.red with one atomic per component.
__global__ void __launch_bounds__(SETUP_THREADS) k_mesh_setup(const MeshUpdate u)
{
  const int k = blockIdx.x * SETUP_THREADS + threadIdx.x;
  double lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
  if (k < u.nTris)
  {
    const int pos = u.triBase + k;
    float v[9];
    for (int j = 0; j < 3; j++)
    {
      const float * p = u.xyz + 3 * (size_t)__ldg(u.idx + 3 * (size_t)k + j);
      v[3 * j] = p[0]; v[3 * j + 1] = p[1]; v[3 * j + 2] = p[2];
    }
    Triangle t;
    setupTriangle(v, t);
    Triangle & bt = u.tris[pos];
    for (int j = 0; j < 3; j++) { bt.v0[j] = t.v0[j]; bt.n[j] = t.n[j]; }
    for (int j = 0; j < 9; j++) bt.ax[j] = t.ax[j];
    if (u.triLeaf)
    {
      TriExtent e;
      triExtent(t.v0, t.ax, e);
      if (e.kappa >= 0.0)
        for (int j = 0; j < 3; j++) { lo[j] = e.lo[j]; hi[j] = e.hi[j]; }
      const int slot = u.triSlot[pos];
      if (slot >= 0 && !(u.far && u.inAlways[pos]))
      {
        float4 * w = u.triLeaf + 3 * (size_t)slot;
        if (u.far && !triBoxed(e))
        {
          // no box holds it from far origins (buildTriBoxes): tested after the walk until the next flatten; an all-zero slot never
          // passes the gate
          u.inAlways[pos] = 1;
          u.triAlways[atomicAdd(&u.header->nTriAlways, 1)] = pos;
          w[0] = w[1] = w[2] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        else
          packTriangle(t, w);
      }
    }
  }
  if (!u.triLeaf) return;
  // block union: warp shuffles, then one warp over the warps' results, then one atomic per component
  __shared__ double sLo[3][SETUP_THREADS / 32], sHi[3][SETUP_THREADS / 32];
  for (int j = 0; j < 3; j++)
    for (int o = 16; o > 0; o >>= 1)
    {
      lo[j] = dmin(lo[j], __shfl_xor_sync(0xFFFFFFFFu, lo[j], o));
      hi[j] = dmax(hi[j], __shfl_xor_sync(0xFFFFFFFFu, hi[j], o));
    }
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  if (lane == 0)
    for (int j = 0; j < 3; j++) { sLo[j][warp] = lo[j]; sHi[j][warp] = hi[j]; }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int j = 0; j < 3; j++)
    {
      double l = sLo[j][0], h = sHi[j][0];
      for (int w = 1; w < SETUP_THREADS / 32; w++) { l = dmin(l, sLo[j][w]); h = dmax(h, sHi[j][w]); }
      if (l <= h)
      {
        atomicMin(u.red + j, orderedCode(l));
        atomicMax(u.red + 3 + j, orderedCode(h));
      }
    }
}

// One thread per leaf: the boxes of all the leaf's triangles from their slot records (the margins of every triangle depend on R), their
// union into the parent pair node (xyz lanes only: the w lanes hold the child refs), then up the tree: the second thread to arrive at a
// pair node unions its two children's boxes and carries on.  The thread that completes the root writes the plane scenes' growth
// terms into the header.
__global__ void __launch_bounds__(REFIT_THREADS) k_tri_refit(const MeshUpdate u)
{
  const int leaf = blockIdx.x * REFIT_THREADS + threadIdx.x;
  if (leaf >= u.nLeaves) return;
  double ulo[3], uhi[3];
  for (int j = 0; j < 3; j++) { ulo[j] = orderedValue(u.red[j]); uhi[j] = orderedValue(u.red[3 + j]); }
  const double R = boxDiagonal(ulo, uhi);
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  double kmax = 0.0;
  for (int s = 0; s < 4; s++)
  {
    const int j = 4 * leaf + s;
    const int pos = u.triPrims[j];
    if (pos < 0 || (u.far && u.inAlways[pos])) continue;
    const float4 * w = u.triLeaf + 3 * (size_t)j;
    const float4 q0 = w[0], q1 = w[1], q2 = w[2];
    const float v0[3] = { q0.x, q0.y, q0.z };
    const float ax[9] = { q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, q0.w, q1.x, q1.y };
    TriExtent e;
    triExtent(v0, ax, e);
    float b[6];
    triBox(e, ulo, uhi, R, u.far, b);
    for (int k = 0; k < 3; k++) { lo[k] = b[k] < lo[k] ? b[k] : lo[k]; hi[k] = hi[k] < b[3 + k] ? b[3 + k] : hi[k]; }
    if (triBoxed(e)) kmax = dmax(kmax, e.kappa);
  }
  if (u.far) atomicMax(u.red + 6, orderedCode(kmax));
  if (!refitClimb(lo, hi, u.leafParent[leaf], u.triPairs, u.pairParent, u.arrive)) return;
  // the root is complete: every leaf's kappa is in red[6]
  if (u.far)
  {
    double U[6];
    for (int j = 0; j < 6; j++) U[j] = orderedValue(u.red[j]);
    roundOutwards(U, u.header->triReach);
    u.header->growT = farGrowthTris(orderedValue(atomicMax(u.red + 6, 0ull)));
  }
}

// One thread per moved sphere: its record into the blob's sphere array (the list walk), its radius, and its leaf slot.
__global__ void __launch_bounds__(SETUP_THREADS) k_sphere_scatter(const SphereUpdate u)
{
  const int k = blockIdx.x * SETUP_THREADS + threadIdx.x;
  if (k >= u.nMoves) return;
  const SphereMove m = u.moves[k];
  u.spheres[m.pos] = m.rec;
  u.radius[m.pos] = m.radius;
  if (u.leafSph) u.leafSph[u.slot[m.pos]] = m.rec;
}

// One thread per leaf: the union of its spheres' boxes (sphereBox at the flatten's R, in slot order as the host build takes them),
// then the climb to the root.  The leaf slots keep the records (unused slots: NaN); only the pair nodes hold boxes.
__global__ void __launch_bounds__(REFIT_THREADS) k_sphere_refit(const SphereUpdate u)
{
  const int leaf = blockIdx.x * REFIT_THREADS + threadIdx.x;
  if (leaf >= u.nLeaves) return;
  float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
  for (int s = 0; s < 4; s++)
  {
    const int j = 4 * leaf + s;
    const int pos = u.prims[j];
    if (pos < 0) continue;
    const float4 q = u.leafSph[j];
    const float c[3] = { q.x, q.y, q.z };
    float blo[3], bhi[3];
    sphereBox(c, u.radius[pos], u.R, blo, bhi);
    for (int k = 0; k < 3; k++) { lo[k] = blo[k] < lo[k] ? blo[k] : lo[k]; hi[k] = hi[k] < bhi[k] ? bhi[k] : hi[k]; }
  }
  refitClimb(lo, hi, u.leafParent[leaf], u.pairs, u.pairParent, u.arrive);
}

} // namespace

int launchSphereUpdate(const SphereUpdate & u, cudaStream_t st)
{
  if (u.nMoves <= 0) return 0;
  k_sphere_scatter<<<(u.nMoves + SETUP_THREADS - 1) / SETUP_THREADS, SETUP_THREADS, 0, st>>>(u);
  if (!u.leafSph) return 1;
  k_sphere_refit<<<(u.nLeaves + REFIT_THREADS - 1) / REFIT_THREADS, REFIT_THREADS, 0, st>>>(u);
  return 2;
}

int launchMeshUpdate(const MeshUpdate & u, cudaStream_t st)
{
  if (u.nTris <= 0) return 0;
  k_mesh_setup<<<(u.nTris + SETUP_THREADS - 1) / SETUP_THREADS, SETUP_THREADS, 0, st>>>(u);
  if (!u.triLeaf) return 1;
  k_tri_refit<<<(u.nLeaves + REFIT_THREADS - 1) / REFIT_THREADS, REFIT_THREADS, 0, st>>>(u);
  return 2;
}

} // namespace rfx
