// device_math_probe.cu — test-only shared library: evaluates the device arithmetic routines of rfx_device.cuh that are not the
// reference's plain IEEE operations (powLikePowf, cubeLikePowf, divExact at its three divisors) on host arrays, so that
// tests/test_device_math.py can hold the compiled device code against exact arithmetic.  Built by that test with the
// product's nvcc flags; not part of the library.  Every call: copy in with cudaMemcpy, one kernel, copy out with cudaMemcpy.
#include <cuda_runtime.h>
#include "../../reflaxman_b200/csrc/rfx_device.cuh"

using namespace rfx;

namespace
{

__global__ void k_pow(int n, const float * x, const float * y, float * out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = powLikePowf(x[i], y[i]);
}

__global__ void k_cube(int n, const float * x, float * out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = cubeLikePowf(x[i]);
}

// which: 0 -> r / 16383.5 (direction draws), 1 -> r / 32767 (additive jitter), 2 -> r / 255 (texels), with the constants the kernels use
__global__ void k_div(int n, int which, const float * r, float * out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (which == 0) out[i] = divExact(r[i], 16383.5f, RFX_RCP_16383_5);
  else if (which == 1) out[i] = divExact(r[i], 32767.0f, RFX_RCP_32767);
  else out[i] = divExact(r[i], 255.0f, RFX_RCP_255);
}

// ins: nin input arrays of n floats; launch(dev inputs, dev out) runs the kernel
template <typename F>
int run(int n, int nin, const float * const * ins, float * out, F launch)
{
  if (n <= 0) return 0;
  const size_t bytes = sizeof(float) * (size_t)n;
  float * d[3] = { nullptr, nullptr, nullptr };
  int rc = 0;
  for (int k = 0; k <= nin && rc == 0; k++)
    if (cudaMalloc(&d[k], bytes) != cudaSuccess) rc = 1;
  for (int k = 0; k < nin && rc == 0; k++)
    if (cudaMemcpy(d[k], ins[k], bytes, cudaMemcpyHostToDevice) != cudaSuccess) rc = 2;
  if (rc == 0)
  {
    launch(d, d[nin], (n + 255) / 256);
    if (cudaGetLastError() != cudaSuccess) rc = 3;
  }
  if (rc == 0 && cudaMemcpy(out, d[nin], bytes, cudaMemcpyDeviceToHost) != cudaSuccess) rc = 4;
  for (int k = 0; k <= nin; k++) cudaFree(d[k]);
  return rc;
}

} // namespace

// the product's flags build with -fvisibility=hidden
#define PROBE_API extern "C" __attribute__((visibility("default")))

PROBE_API int probe_pow(int n, const float * x, const float * y, float * out)
{
  const float * ins[2] = { x, y };
  return run(n, 2, ins, out, [n](float ** d, float * o, int blocks) { k_pow<<<blocks, 256>>>(n, d[0], d[1], o); });
}

PROBE_API int probe_cube(int n, const float * x, float * out)
{
  const float * ins[1] = { x };
  return run(n, 1, ins, out, [n](float ** d, float * o, int blocks) { k_cube<<<blocks, 256>>>(n, d[0], o); });
}

PROBE_API int probe_div(int n, int which, const float * r, float * out)
{
  const float * ins[1] = { r };
  return run(n, 1, ins, out, [n, which](float ** d, float * o, int blocks) { k_div<<<blocks, 256>>>(n, which, d[0], o); });
}
