// lbvh.cuh -- the kernels both device builders run: Morton codes, the binary radix tree (Karras 2012) and the bottom-up box
// fit.  bvh_build_gpu.cu builds geometries with them, bvh_build_ias_gpu.cu the instance level.  Their arithmetic is in
// bvh_rules.h, which the host twin of the instance-level rebuild (accel_host.cpp) shares.
#pragma once

#include "rtc_internal.h"
#include "bvh_rules.h"

namespace {

constexpr int kLbvhBlock = 256;

// ---- float atomics through the order-preserving integer image -------------------------------------------------
__device__ __forceinline__ void atomicMinF(float* addr, float v)
{
  if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
  else           atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomicMaxF(float* addr, float v)
{
  if (v >= 0.0f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else           atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__global__ void __launch_bounds__(kLbvhBlock)
k_morton(const float4* __restrict__ triLo, const float4* __restrict__ triHi, uint32_t n, const float* __restrict__ sceneBox,
         unsigned long long* __restrict__ keys, uint32_t* __restrict__ order)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  keys[t] = lbvh_morton(triLo[t], triHi[t], sceneBox);
  order[t] = t;
}

__global__ void __launch_bounds__(kLbvhBlock)
k_radix_tree(const unsigned long long* __restrict__ keys, int n, int2* __restrict__ child, int* __restrict__ parent, int2* __restrict__ range)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  lbvh_radix_node(keys, n, i, child, parent, range);
}

__global__ void __launch_bounds__(kLbvhBlock)
k_fit_boxes(int n, const uint32_t* __restrict__ order, const float4* __restrict__ triLo, const float4* __restrict__ triHi,
            const int2* __restrict__ child, const int* __restrict__ parent, float4* __restrict__ boxLo, float4* __restrict__ boxHi,
            uint32_t* __restrict__ flags)
{
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const uint32_t t = order[p];
  float4 lo = triLo[t], hi = triHi[t];
  int node = n - 1 + p;
  boxLo[node] = lo; boxHi[node] = hi;
  if (n == 1) return;
  __threadfence();
  node = parent[node];
  while (node >= 0)
  {
    if (atomicAdd(flags + node, 1u) == 0u) return;      // the second child to arrive carries on
    __threadfence();
    const int2 c = child[node];
    const volatile float4* vLo = boxLo; const volatile float4* vHi = boxHi;
    const float lx = fminf(vLo[c.x].x, vLo[c.y].x), ly = fminf(vLo[c.x].y, vLo[c.y].y), lz = fminf(vLo[c.x].z, vLo[c.y].z);
    const float hx = fmaxf(vHi[c.x].x, vHi[c.y].x), hy = fmaxf(vHi[c.x].y, vHi[c.y].y), hz = fmaxf(vHi[c.x].z, vHi[c.y].z);
    boxLo[node] = make_float4(lx, ly, lz, 0.0f); boxHi[node] = make_float4(hx, hy, hz, 0.0f);
    __threadfence();
    node = parent[node];
  }
}

} // namespace
