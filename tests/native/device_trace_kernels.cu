// tests/native/device_trace_kernels.cu -- TEST INFRASTRUCTURE: user kernels that call the device-side queries of
// include/rtc_device.cuh, as a caller of the library writes them (compiled with -Iinclude only), with C launchers for ctypes.
// Built by tests/test_gpu_device_trace.py (default flags and -fmad=false) and by tools/device_trace_bench.py.
#include "rtc_device.cuh"

namespace {

// One query per thread.  masks / flags: per ray (null: `mask` / `flags` for every ray).  oddOnly: even threads return at once,
// so every warp runs the query on half of its lanes.  status: per ray, or null.  BIG: compiled for 1024-thread blocks.
template <bool ANY, bool BIG>
__global__ void __launch_bounds__(BIG ? 1024 : 256)
k_query(uint64_t top, const rtc_ray* __restrict__ rays, uint32_t n, const uint32_t* __restrict__ masks, const uint32_t* __restrict__ flags,
        uint32_t mask, uint32_t fl, void* __restrict__ out, int* __restrict__ status, int oddOnly)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (oddOnly && !(i & 1u))) return;
  const rtc_ray ray = rays[i];
  const uint32_t m = masks ? masks[i] : mask, f = flags ? flags[i] : fl;
  int s;
  if (ANY) s = rtc_device_trace_any(top, ray, static_cast<uint32_t*>(out) + i, m, f);
  else     s = rtc_device_trace_closest(top, ray, static_cast<rtc_hit*>(out) + i, m, f);
  if (status) status[i] = s;
}

// Ray k of the ambient-occlusion rays of pixel p: from the primary hit point, in a direction hashed from (p, k), over
// (1e-3, radius).  A primary miss gives an empty interval.  Rounding pinned with intrinsics, so that the fused kernel and the
// ray-writing kernel compute the same bits whatever the compiler contracts.
__device__ __forceinline__ uint32_t hash32(uint32_t x)
{
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}

__device__ __forceinline__ rtc_ray ao_ray(const rtc_ray& primary, const rtc_hit& hit, uint32_t p, uint32_t k, float radius)
{
  rtc_ray r;
  const float t = hit.inst != 0xffffffffu ? hit.t : 0.0f;
  r.ox = __fmaf_rn(t, primary.dx, primary.ox); r.oy = __fmaf_rn(t, primary.dy, primary.oy); r.oz = __fmaf_rn(t, primary.dz, primary.oz);
  const uint32_t h0 = hash32(p * 8u + k), h1 = hash32(h0 ^ 0x9e3779b9u), h2 = hash32(h1 ^ 0x85ebca6bu);
  r.dx = __fsub_rn(__fmul_rn((float)(h0 >> 8), 0x1p-23f), 1.0f);
  r.dy = __fsub_rn(__fmul_rn((float)(h1 >> 8), 0x1p-23f), 1.0f);
  r.dz = __fsub_rn(__fmul_rn((float)(h2 >> 8), 0x1p-23f), 1.0f);
  r.tmin = 1e-3f;
  r.tmax = hit.inst != 0xffffffffu ? radius : -1.0f;
  return r;
}

// Fused: primary closest hit, `samples` occlusion rays, the count reduced in a register.
__global__ void __launch_bounds__(256)
k_ao_fused(uint64_t top, const rtc_ray* __restrict__ primary, uint32_t n, uint32_t samples, float radius, rtc_hit* __restrict__ hits,
           uint32_t* __restrict__ occludedCount)
{
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const rtc_ray ray = primary[p];
  rtc_hit hit;
  rtc_device_trace_closest(top, ray, &hit);
  uint32_t count = 0;
  if (hit.inst != 0xffffffffu)
    for (uint32_t k = 0; k < samples; ++k)
    {
      uint32_t occ;
      rtc_device_trace_any(top, ao_ray(ray, hit, p, k, radius), &occ);
      count += occ;
    }
  hits[p] = hit;
  occludedCount[p] = count;
}

// The three-call pipeline's middle and last steps: the occlusion rays of every pixel, and the per-pixel count of occluded ones.
__global__ void k_ao_rays(const rtc_ray* __restrict__ primary, const rtc_hit* __restrict__ hits, uint32_t n, uint32_t samples, float radius,
                          rtc_ray* __restrict__ aoRays)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * samples) return;
  const uint32_t p = i / samples, k = i - p * samples;
  aoRays[i] = ao_ray(primary[p], hits[p], p, k, radius);
}

__global__ void k_ao_reduce(const uint32_t* __restrict__ occluded, uint32_t n, uint32_t samples, uint32_t* __restrict__ occludedCount)
{
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  uint32_t count = 0;
  for (uint32_t k = 0; k < samples; ++k) count += occluded[(size_t)p * samples + k];
  occludedCount[p] = count;
}

// this translation unit's overflow counter (rtc_device.cuh)
__global__ void k_read_overflows(unsigned int* out) { *out = rtc_device_stack_overflows; }

uint32_t blocks(uint64_t n, int block) { return (uint32_t)((n + (uint64_t)block - 1) / (uint64_t)block); }

} // namespace

extern "C" {

// any: 0 closest (out = rtc_hit[n]), 1 any (out = uint32[n]); block: threads per block (1024 takes the kernel built for it)
int dt_query(int any, uint64_t top, uint64_t rays, uint32_t n, uint64_t masks, uint64_t flags, uint32_t mask, uint32_t fl, uint64_t out,
             uint64_t status, int block, int oddOnly, uint64_t stream)
{
  if (n == 0) return 0;
  cudaStream_t s = reinterpret_cast<cudaStream_t>((uintptr_t)stream);
  const rtc_ray* r = reinterpret_cast<const rtc_ray*>((uintptr_t)rays);
  const uint32_t* m = reinterpret_cast<const uint32_t*>((uintptr_t)masks);
  const uint32_t* f = reinterpret_cast<const uint32_t*>((uintptr_t)flags);
  void* o = reinterpret_cast<void*>((uintptr_t)out);
  int* st = reinterpret_cast<int*>((uintptr_t)status);
  if (block > 256)
  {
    if (any) k_query<true, true><<<blocks(n, block), block, 0, s>>>(top, r, n, m, f, mask, fl, o, st, oddOnly);
    else     k_query<false, true><<<blocks(n, block), block, 0, s>>>(top, r, n, m, f, mask, fl, o, st, oddOnly);
  }
  else
  {
    if (any) k_query<true, false><<<blocks(n, block), block, 0, s>>>(top, r, n, m, f, mask, fl, o, st, oddOnly);
    else     k_query<false, false><<<blocks(n, block), block, 0, s>>>(top, r, n, m, f, mask, fl, o, st, oddOnly);
  }
  return (int)cudaGetLastError();
}

int dt_ao_fused(uint64_t top, uint64_t primary, uint32_t n, uint32_t samples, float radius, uint64_t hits, uint64_t counts, uint64_t stream)
{
  if (n == 0) return 0;
  k_ao_fused<<<blocks(n, 128), 128, 0, reinterpret_cast<cudaStream_t>((uintptr_t)stream)>>>(
      top, reinterpret_cast<const rtc_ray*>((uintptr_t)primary), n, samples, radius, reinterpret_cast<rtc_hit*>((uintptr_t)hits),
      reinterpret_cast<uint32_t*>((uintptr_t)counts));
  return (int)cudaGetLastError();
}

int dt_ao_rays(uint64_t primary, uint64_t hits, uint32_t n, uint32_t samples, float radius, uint64_t aoRays, uint64_t stream)
{
  if (n == 0) return 0;
  k_ao_rays<<<blocks((uint64_t)n * samples, 256), 256, 0, reinterpret_cast<cudaStream_t>((uintptr_t)stream)>>>(
      reinterpret_cast<const rtc_ray*>((uintptr_t)primary), reinterpret_cast<const rtc_hit*>((uintptr_t)hits), n, samples, radius,
      reinterpret_cast<rtc_ray*>((uintptr_t)aoRays));
  return (int)cudaGetLastError();
}

int dt_ao_reduce(uint64_t occluded, uint32_t n, uint32_t samples, uint64_t counts, uint64_t stream)
{
  if (n == 0) return 0;
  k_ao_reduce<<<blocks(n, 256), 256, 0, reinterpret_cast<cudaStream_t>((uintptr_t)stream)>>>(
      reinterpret_cast<const uint32_t*>((uintptr_t)occluded), n, samples, reinterpret_cast<uint32_t*>((uintptr_t)counts));
  return (int)cudaGetLastError();
}

// rtc_device_stack_overflows of this module into the device word at `out`
int dt_stack_overflows(uint64_t out, uint64_t stream)
{
  k_read_overflows<<<1, 1, 0, reinterpret_cast<cudaStream_t>((uintptr_t)stream)>>>(reinterpret_cast<unsigned int*>((uintptr_t)out));
  return (int)cudaGetLastError();
}

} // extern "C"
