// tests/native/device_anyhit_kernels.cu -- TEST INFRASTRUCTURE: user kernels that call the any-hit queries of
// include/rtc_device.cuh, as a caller of the library writes them (plain lambdas, compiled with -Iinclude only), with C launchers
// for ctypes.  Built by tests/test_gpu_device_anyhit.py (default flags and -fmad=false) and by tools/device_anyhit_bench.py.
#include "rtc_device.cuh"
#include "anyhit_predicates.h"

extern "C" {
// one launch of k_anyhit; null pointers are not read or written (masks / flags null: `mask` / `fl` for every ray; p0 / p1 null: 0)
struct da_args
{
  uint64_t top;
  const rtc_ray* rays;
  const uint32_t* masks;
  const uint32_t* flags;
  const uint32_t* p0;
  const uint32_t* p1;
  void* out;                 // closest: rtc_hit[n]; any: uint32[n]
  int* status;
  uint32_t* calls;           // callback calls per ray
  ahp_record* records;       // the first k calls of ray i at records[i * k]
  uint32_t* digest;          // count, sum, XOR of the calls of ray i at digest[3 i]
  uint32_t n, mask, fl, k;
  int pred, end, oddOnly, pad;
};
}

namespace {

// One query per thread with a recording callback that decides with anyhit_predicates.h.  oddOnly: even threads return at once.
template <bool ANY, bool BIG>
__global__ void __launch_bounds__(BIG ? 1024 : 256) k_anyhit(const da_args a)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n || (a.oddOnly && !(i & 1u))) return;
  const rtc_ray ray = a.rays[i];
  const uint32_t m = a.masks ? a.masks[i] : a.mask, f = a.flags ? a.flags[i] : a.fl;
  const uint32_t q0 = a.p0 ? a.p0[i] : 0u, q1 = a.p1 ? a.p1[i] : 0u;
  uint32_t count = 0, d[3] = { 0u, 0u, 0u };
  auto anyHit = [&](const rtc_candidate& c) {
    if (a.records && count < a.k)
    {
      const ahp_record r = { c.t, c.u, c.v, c.inst, c.prim, c.frontFacing };
      a.records[(size_t)i * a.k + count] = r;
    }
    ++count;
    ahp_digest_add(d, c.t, c.u, c.v, c.inst, c.prim, c.frontFacing);
    return ahp_decide(a.pred, c.t, c.u, c.v, c.inst, c.prim, c.frontFacing, q0, q1, a.end);
  };
  int s;
  if (ANY) s = rtc_device_trace_any_anyhit(a.top, ray, static_cast<uint32_t*>(a.out) + i, anyHit, m, f);
  else     s = rtc_device_trace_closest_anyhit(a.top, ray, static_cast<rtc_hit*>(a.out) + i, anyHit, m, f);
  if (a.status) a.status[i] = s;
  if (a.calls) a.calls[i] = count;
  if (a.digest) { a.digest[3 * i] = d[0]; a.digest[3 * i + 1] = d[1]; a.digest[3 * i + 2] = d[2]; }
}

// The kernels of the measurements, without recording.  MODE 0: rtc_device_trace_closest / _any.  1: the always-accept callback.
// 2: the alpha test of anyhit_predicates.h (alpha = transparent triangles per 256).  3 (ANY only): every candidate, ignored,
// counted and digested (out = count per ray, digest = sum and XOR per ray).
template <bool ANY, int MODE>
__global__ void __launch_bounds__(256) k_lean(uint64_t top, const rtc_ray* __restrict__ rays, uint32_t n, uint32_t alpha, void* __restrict__ out,
                                              uint32_t* __restrict__ digest)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const rtc_ray ray = rays[i];
  rtc_hit* hit = static_cast<rtc_hit*>(out) + i;
  uint32_t* occ = static_cast<uint32_t*>(out) + i;
  if (MODE == 0)
  {
    if (ANY) rtc_device_trace_any(top, ray, occ);
    else     rtc_device_trace_closest(top, ray, hit);
  }
  else if (MODE == 1)
  {
    auto accept = [](const rtc_candidate&) { return true; };
    if (ANY) rtc_device_trace_any_anyhit(top, ray, occ, accept);
    else     rtc_device_trace_closest_anyhit(top, ray, hit, accept);
  }
  else if (MODE == 2)
  {
    auto opaque = [&](const rtc_candidate& c) { return ahp_alpha(c.inst, c.prim, c.u, c.v, alpha) != 0; };
    if (ANY) rtc_device_trace_any_anyhit(top, ray, occ, opaque);
    else     rtc_device_trace_closest_anyhit(top, ray, hit, opaque);
  }
  else
  {
    uint32_t d[3] = { 0u, 0u, 0u }, o;
    rtc_device_trace_any_anyhit(top, ray, &o, [&](const rtc_candidate& c) {
      ahp_digest_add(d, c.t, c.u, c.v, c.inst, c.prim, c.frontFacing);
      return RTC_ANYHIT_IGNORE;
    });
    *occ = d[0];
    digest[2 * i] = d[1]; digest[2 * i + 1] = d[2];
  }
}

// What a caller writes without callbacks: trace again from tmin = t of every transparent hit until an opaque hit or a miss.
// Candidates at exactly the t of a rejected hit are skipped, because the next query needs t > tmin.
__global__ void __launch_bounds__(256) k_alpha_restart(uint64_t top, const rtc_ray* __restrict__ rays, uint32_t n, uint32_t alpha,
                                                       rtc_hit* __restrict__ hits, uint32_t* __restrict__ restarts)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rtc_ray ray = rays[i];
  rtc_hit h;
  uint32_t k = 0;
  for (;;)
  {
    rtc_device_trace_closest(top, ray, &h);
    if (h.inst == 0xffffffffu || ahp_alpha(h.inst, h.prim, h.u, h.v, alpha)) break;
    ray.tmin = h.t;
    ++k;
  }
  hits[i] = h;
  restarts[i] = k;
}

// Ray from the hit of `primary` in a direction hashed from p (as the ambient-occlusion rays of device_trace_kernels.cu), over
// (tmin, tmax); a primary miss gives an empty interval.
__device__ __forceinline__ rtc_ray hashed_ray(const rtc_ray& primary, const rtc_hit& hit, uint32_t p, float tmin, float tmax)
{
  rtc_ray r;
  const float t = hit.inst != 0xffffffffu ? hit.t : 0.0f;
  r.ox = __fmaf_rn(t, primary.dx, primary.ox); r.oy = __fmaf_rn(t, primary.dy, primary.oy); r.oz = __fmaf_rn(t, primary.dz, primary.oz);
  const uint32_t h0 = ahp_hash(p * 8u), h1 = ahp_hash(h0 ^ 0x9e3779b9u), h2 = ahp_hash(h1 ^ 0x85ebca6bu);
  r.dx = __fsub_rn(__fmul_rn((float)(h0 >> 8), 0x1p-23f), 1.0f);
  r.dy = __fsub_rn(__fmul_rn((float)(h1 >> 8), 0x1p-23f), 1.0f);
  r.dz = __fsub_rn(__fmul_rn((float)(h2 >> 8), 0x1p-23f), 1.0f);
  r.tmin = tmin;
  r.tmax = hit.inst != 0xffffffffu ? tmax : -1.0f;
  return r;
}

__global__ void k_secondary_rays(const rtc_ray* __restrict__ primary, const rtc_hit* __restrict__ hits, uint32_t n, rtc_ray* __restrict__ out)
{
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) out[p] = hashed_ray(primary[p], hits[p], p, 1e-3f, 1e27f);
}

// Self-intersection avoidance by identity: the primary hit, then a ray from that point with tmin = 0 that ignores the
// primary's triangle instead of relying on an epsilon.
__global__ void __launch_bounds__(256) k_self_skip(uint64_t top, const rtc_ray* __restrict__ primary, uint32_t n, rtc_hit* __restrict__ primaryHits,
                                                   rtc_ray* __restrict__ secondary, rtc_hit* __restrict__ secondaryHits)
{
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const rtc_ray ray = primary[p];
  rtc_hit hit;
  rtc_device_trace_closest(top, ray, &hit);
  const rtc_ray r = hashed_ray(ray, hit, p, 0.0f, 1e27f);
  rtc_hit second;
  rtc_device_trace_closest_anyhit(top, r, &second, [&](const rtc_candidate& c) { return !(c.inst == hit.inst && c.prim == hit.prim); });
  primaryHits[p] = hit;
  secondary[p] = r;
  secondaryHits[p] = second;
}

// this translation unit's overflow counter (rtc_device.cuh)
__global__ void k_read_overflows(unsigned int* out) { *out = rtc_device_stack_overflows; }

uint32_t blocks(uint64_t n, int block) { return (uint32_t)((n + (uint64_t)block - 1) / (uint64_t)block); }
cudaStream_t as_stream(uint64_t s) { return reinterpret_cast<cudaStream_t>((uintptr_t)s); }
template <class T> T* ptr(uint64_t p) { return reinterpret_cast<T*>((uintptr_t)p); }

} // namespace

extern "C" {

// any: 0 closest, 1 any; block: threads per block (above 256 takes the kernel built for 1024)
int da_query(int any, const da_args* a, int block, uint64_t stream)
{
  if (a->n == 0) return 0;
  const cudaStream_t s = as_stream(stream);
  if (block > 256)
  {
    if (any) k_anyhit<true, true><<<blocks(a->n, block), block, 0, s>>>(*a);
    else     k_anyhit<false, true><<<blocks(a->n, block), block, 0, s>>>(*a);
  }
  else
  {
    if (any) k_anyhit<true, false><<<blocks(a->n, block), block, 0, s>>>(*a);
    else     k_anyhit<false, false><<<blocks(a->n, block), block, 0, s>>>(*a);
  }
  return (int)cudaGetLastError();
}

// mode: k_lean's MODE
int da_lean(int any, int mode, uint64_t top, uint64_t rays, uint32_t n, uint32_t alpha, uint64_t out, uint64_t digest, uint64_t stream)
{
  if (n == 0) return 0;
  const cudaStream_t s = as_stream(stream);
  const rtc_ray* r = ptr<const rtc_ray>(rays);
  void* o = ptr<void>(out);
  uint32_t* d = ptr<uint32_t>(digest);
  const uint32_t g = blocks(n, 128);
  switch (any * 4 + mode)
  {
  case 0: k_lean<false, 0><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  case 1: k_lean<false, 1><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  case 2: k_lean<false, 2><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  case 4: k_lean<true, 0><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  case 5: k_lean<true, 1><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  case 6: k_lean<true, 2><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  case 7: k_lean<true, 3><<<g, 128, 0, s>>>(top, r, n, alpha, o, d); break;
  default: return -1;
  }
  return (int)cudaGetLastError();
}

int da_alpha_restart(uint64_t top, uint64_t rays, uint32_t n, uint32_t alpha, uint64_t hits, uint64_t restarts, uint64_t stream)
{
  if (n == 0) return 0;
  k_alpha_restart<<<blocks(n, 128), 128, 0, as_stream(stream)>>>(top, ptr<const rtc_ray>(rays), n, alpha, ptr<rtc_hit>(hits), ptr<uint32_t>(restarts));
  return (int)cudaGetLastError();
}

int da_secondary_rays(uint64_t primary, uint64_t hits, uint32_t n, uint64_t out, uint64_t stream)
{
  if (n == 0) return 0;
  k_secondary_rays<<<blocks(n, 256), 256, 0, as_stream(stream)>>>(ptr<const rtc_ray>(primary), ptr<const rtc_hit>(hits), n, ptr<rtc_ray>(out));
  return (int)cudaGetLastError();
}

int da_self_skip(uint64_t top, uint64_t primary, uint32_t n, uint64_t primaryHits, uint64_t secondary, uint64_t secondaryHits, uint64_t stream)
{
  if (n == 0) return 0;
  k_self_skip<<<blocks(n, 128), 128, 0, as_stream(stream)>>>(top, ptr<const rtc_ray>(primary), n, ptr<rtc_hit>(primaryHits), ptr<rtc_ray>(secondary),
                                                             ptr<rtc_hit>(secondaryHits));
  return (int)cudaGetLastError();
}

int da_stack_overflows(uint64_t out, uint64_t stream)
{
  k_read_overflows<<<1, 1, 0, as_stream(stream)>>>(ptr<unsigned int>(out));
  return (int)cudaGetLastError();
}

} // extern "C"
