// kernels_trace.cu -- the traversal kernels: ray queries (rtc_trace_*), and the wavefront integrator's
// extend (closest hit of the radiance-ray queue) and connect (any hit of the shadow-ray queue).
// All of them are persistent-warp kernels over trace_stream() (trace.cuh, one ray per lane): one CTA of 128 threads per
// resident slot, rays handed out through a device-side cursor.
// Built for sm_100a with FMA contraction ON: only the box tests may contract; the intersector in
// trace.cuh pins its own rounding with intrinsics.
#include "trace.cuh"

namespace {

constexpr int kTraceBlock = 128;

// ---- ray sources / hit sinks (stateless: the per-ray word `tag` travels with the ray) -------------------------------

// rtc_trace_closest: AoS rays in, rtc_hit out
struct QueryClosest
{
  const float4* __restrict__ rays; rtc_hit* __restrict__ hits;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& tag) const { tag = i; o = __ldg(rays + 2 * (size_t)i); d = __ldg(rays + 2 * (size_t)i + 1); return true; }
  __device__ __forceinline__ void store(uint32_t tag, const TraceHit& h) const
  {
    rtc_hit out; out.t = h.t; out.u = h.u; out.v = h.v; out.inst = h.inst; out.prim = h.prim;
    hits[tag] = out;
  }
};

// rtc_trace_any: AoS rays in, one uint32 per ray out
struct QueryAny
{
  const float4* __restrict__ rays; uint32_t* __restrict__ occluded;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& tag) const { tag = i; o = __ldg(rays + 2 * (size_t)i); d = __ldg(rays + 2 * (size_t)i + 1); return true; }
  __device__ __forceinline__ void store(uint32_t tag, const TraceHit& h) const { occluded[tag] = h.inst != 0xffffffffu ? 1u : 0u; }
};

// rtc_trace_count: rays in, nothing out (the counters are the result)
struct QueryCount
{
  const float4* __restrict__ rays;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& tag) const { tag = i; o = __ldg(rays + 2 * (size_t)i); d = __ldg(rays + 2 * (size_t)i + 1); return true; }
  __device__ __forceinline__ void store(uint32_t, const TraceHit&) const {}
};

// extend: queue of path ids -> SoA radiance rays; hit record per path (raygeneration.cu:84-89 optixTrace RADIANCE)
struct ExtendPaths
{
  const uint32_t* __restrict__ queue; const float4* __restrict__ rayOrg; const float4* __restrict__ rayDir;
  float4* __restrict__ hit; uint32_t* __restrict__ hitInst;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& path) const { path = queue[i]; o = rayOrg[path]; d = rayDir[path]; return true; }
  __device__ __forceinline__ void store(uint32_t path, const TraceHit& h) const
  {
    __stcs(hit + path, make_float4(h.t, h.u, h.v, __uint_as_float(h.prim)));
    __stcs(hitInst + path, h.inst);
  }
};

// connect: queue of path ids -> SoA shadow rays (closesthit.cu:281-300 + anyhit.cu:84-91); an unoccluded ray adds its
// pre-multiplied contribution to the path radiance (each path has at most one shadow ray in flight: no race).
struct ConnectPaths
{
  const uint32_t* __restrict__ queue; const float4* __restrict__ shadowOrg; const float4* __restrict__ shadowDir;
  const float4* __restrict__ contrib; float4* __restrict__ radiance;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& path) const { path = queue[i]; o = shadowOrg[path]; d = shadowDir[path]; return true; }
  __device__ __forceinline__ void store(uint32_t path, const TraceHit& h) const
  {
    if (h.inst == 0xffffffffu)
    {
      const float4 c = __ldcs(contrib + path);
      float4 L = __ldcs(radiance + path);
      L.x = __fadd_rn(L.x, c.x); L.y = __fadd_rn(L.y, c.y); L.z = __fadd_rn(L.z, c.z);
      __stcs(radiance + path, L);
    }
  }
};

// ---- ordered any-hit processing (scenes with cutout materials only; anyhit.cu:46-132) ----------------------------------
// The closest candidate of a ray is found by the normal kernels; when the any-hit program ignores it (k_cutout_radiance /
// k_cutout_shadow in kernels_shade.cu), the ray is traced again for the next candidate AFTER the ignored one.  The ignored
// hit sits in hit[path] / hitInst[path] and is the skip key; tmin moves up to just below its t (ties are resolved by the key).

// radiance ray of a path, again, past the candidate in hit[path]
struct ExtendPathsAfter
{
  const uint32_t* __restrict__ queue; const float4* __restrict__ rayOrg; const float4* __restrict__ rayDir;
  float4* __restrict__ hit; uint32_t* __restrict__ hitInst;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& path) const
  {
    path = queue[i]; o = rayOrg[path]; d = rayDir[path];
    o.w = fmaxf(o.w, __uint_as_float(__float_as_uint(hit[path].x) - 1u));      // previous t > tmin > 0
    return true;
  }
  __device__ __forceinline__ void skip_key(uint32_t path, float& t, uint32_t& inst, uint32_t& prim) const
  {
    const float4 prev = hit[path];
    t = prev.x; inst = hitInst[path]; prim = __float_as_uint(prev.w);
  }
  __device__ __forceinline__ void store(uint32_t path, const TraceHit& h) const
  {
    hit[path] = make_float4(h.t, h.u, h.v, __uint_as_float(h.prim));
    hitInst[path] = h.inst;
  }
};

// shadow ray of a path as a CLOSEST-hit query (first candidate, or the next one after hit[path] when AFTER)
template <bool AFTER>
struct ConnectClosest
{
  const uint32_t* __restrict__ queue; const float4* __restrict__ shadowOrg; const float4* __restrict__ shadowDir;
  float4* __restrict__ hit; uint32_t* __restrict__ hitInst;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& path) const
  {
    path = queue[i]; o = shadowOrg[path]; d = shadowDir[path];
    if (AFTER) o.w = fmaxf(o.w, __uint_as_float(__float_as_uint(hit[path].x) - 1u));
    return true;
  }
  __device__ __forceinline__ void skip_key(uint32_t path, float& t, uint32_t& inst, uint32_t& prim) const
  {
    const float4 prev = hit[path];
    t = prev.x; inst = hitInst[path]; prim = __float_as_uint(prev.w);
  }
  __device__ __forceinline__ void store(uint32_t path, const TraceHit& h) const
  {
    hit[path] = make_float4(h.t, h.u, h.v, __uint_as_float(h.prim));
    hitInst[path] = h.inst;
  }
};

// ---- kernels ---------------------------------------------------------------------------------------------------------

// TRICAP: the capped schedules of the triangle tests (trace.cuh Traversal::step); 1 and 2 are instantiated for the timed kernels only.
template <bool ANY, bool COUNT, class Policy, bool SKIP = false, int TRICAP = 0>
__global__ void __launch_bounds__(kTraceBlock, SKIP ? 4 : RTC_TRACE_MIN_BLOCKS)
k_trace(const SceneDesc sc, const Policy policy, uint32_t n, const uint32_t* __restrict__ nPtr, uint32_t* __restrict__ cursor,
        unsigned long long* __restrict__ counts)
{
  __shared__ uint2 smem[RTC_SM_STACK * kTraceBlock + (RTC_SM_RAY_WORDS * kTraceBlock + 1) / 2];     // stack columns, then the float columns (trace.cuh smRay)
  const uint32_t count = nPtr ? *nPtr : n;
  trace_stream<ANY, COUNT, kTraceBlock, SKIP, TRICAP>(sc, count, cursor, policy, smem, counts);
}

template <bool ANY, bool COUNT, class Policy, bool SKIP>
int launch_k_trace(rtc_context* ctx, const SceneDesc* scene, const Policy& p, uint32_t n, const uint32_t* nPtr, uint32_t* cursor, unsigned long long* counts)
{
  if (!COUNT && !SKIP && ctx->traceSchedule == RTC_SCHEDULE_ONE_TRI)
  {
    // the counting kernels and the ordered any-hit re-traces keep the one schedule: their per-ray results do not depend on it
    k_trace<ANY, false, Policy, false, 1><<<ctx->numSMs * RTC_TRACE_MIN_BLOCKS, kTraceBlock, 0, ctx->stream>>>(*scene, p, n, nPtr, cursor, counts);
  }
  else if (!COUNT && !SKIP && ctx->traceSchedule == RTC_SCHEDULE_TWO_TRI)
  {
    k_trace<ANY, false, Policy, false, 2><<<ctx->numSMs * RTC_TRACE_MIN_BLOCKS, kTraceBlock, 0, ctx->stream>>>(*scene, p, n, nPtr, cursor, counts);
  }
  else
  {
    k_trace<ANY, COUNT, Policy, SKIP><<<ctx->numSMs * RTC_TRACE_MIN_BLOCKS, kTraceBlock, 0, ctx->stream>>>(*scene, p, n, nPtr, cursor, counts);
  }
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

} // namespace

// With lazy module loading a kernel is loaded at its first launch; the schedule tuner must not time that.
void preload_capped_trace_kernels()
{
  cudaFuncAttributes attr;
  cudaFuncGetAttributes(&attr, k_trace<false, false, ExtendPaths, false, 1>);
  cudaFuncGetAttributes(&attr, k_trace<true, false, ConnectPaths, false, 1>);
  cudaFuncGetAttributes(&attr, k_trace<false, false, ExtendPaths, false, 2>);
  cudaFuncGetAttributes(&attr, k_trace<true, false, ConnectPaths, false, 2>);
  cudaGetLastError();
}

int launch_trace_closest(rtc_context* ctx, const SceneDesc* scene, const rtc_ray* rays, uint64_t n, rtc_hit* hits)
{
  if (n == 0) return 0;
  if (n > 0xfffffff0ull) RTC_FAIL("more than 2^32 rays in one call");
  RTC_CUDA(cudaMemsetAsync(ctx->d_cursor, 0, sizeof(uint32_t), ctx->stream));
  QueryClosest p = { reinterpret_cast<const float4*>(rays), hits };
  return launch_k_trace<false, false, QueryClosest, false>(ctx, scene, p, (uint32_t)n, nullptr, ctx->d_cursor, nullptr);
}

int launch_trace_any(rtc_context* ctx, const SceneDesc* scene, const rtc_ray* rays, uint64_t n, uint32_t* occluded)
{
  if (n == 0) return 0;
  if (n > 0xfffffff0ull) RTC_FAIL("more than 2^32 rays in one call");
  RTC_CUDA(cudaMemsetAsync(ctx->d_cursor, 0, sizeof(uint32_t), ctx->stream));
  QueryAny p = { reinterpret_cast<const float4*>(rays), occluded };
  return launch_k_trace<true, false, QueryAny, false>(ctx, scene, p, (uint32_t)n, nullptr, ctx->d_cursor, nullptr);
}

int launch_trace_count(rtc_context* ctx, const SceneDesc* scene, const rtc_ray* rays, uint64_t n, int anyHit, unsigned long long* d_counts)
{
  if (n == 0) return 0;
  if (n > 0xfffffff0ull) RTC_FAIL("more than 2^32 rays in one call");
  RTC_CUDA(cudaMemsetAsync(ctx->d_cursor, 0, sizeof(uint32_t), ctx->stream));
  QueryCount p = { reinterpret_cast<const float4*>(rays) };
  if (anyHit) return launch_k_trace<true, true, QueryCount, false>(ctx, scene, p, (uint32_t)n, nullptr, ctx->d_cursor, d_counts);
  return launch_k_trace<false, true, QueryCount, false>(ctx, scene, p, (uint32_t)n, nullptr, ctx->d_cursor, d_counts);
}

int launch_extend(rtc_context* ctx, const SceneDesc* scene, const WavefrontBuffers& wf, const uint32_t* queue, const uint32_t* count,
                  uint32_t* cursor, bool countWork)
{
  if (int rc = profile_begin(ctx, RTC_KERNEL_EXTEND)) return rc;
  ExtendPaths p = { queue, wf.rayOrg, wf.rayDir, wf.hit, wf.hitInst };
  if (int rc = countWork ? launch_k_trace<false, true, ExtendPaths, false>(ctx, scene, p, 0u, count, cursor, ctx->d_launchCounts)
                         : launch_k_trace<false, false, ExtendPaths, false>(ctx, scene, p, 0u, count, cursor, nullptr)) return rc;
  return profile_end(ctx);
}

int launch_connect(rtc_context* ctx, const SceneDesc* scene, const WavefrontBuffers& wf, const uint32_t* count, uint32_t* cursor, bool countWork)
{
  if (int rc = profile_begin(ctx, RTC_KERNEL_CONNECT)) return rc;
  ConnectPaths p = { wf.shadowQueue, wf.shadowOrg, wf.shadowDir, wf.shadowContrib, wf.radiance };
  if (int rc = countWork ? launch_k_trace<true, true, ConnectPaths, false>(ctx, scene, p, 0u, count, cursor, ctx->d_launchCounts + kTraceCountWords)
                         : launch_k_trace<true, false, ConnectPaths, false>(ctx, scene, p, 0u, count, cursor, nullptr)) return rc;
  return profile_end(ctx);
}

// Re-trace of the radiance rays in `queue` past their ignored candidate (see ExtendPathsAfter).
int launch_extend_after(rtc_context* ctx, const SceneDesc* scene, const WavefrontBuffers& wf, const uint32_t* queue, const uint32_t* count, uint32_t* cursor)
{
  if (int rc = profile_begin(ctx, RTC_KERNEL_EXTEND)) return rc;
  ExtendPathsAfter p = { queue, wf.rayOrg, wf.rayDir, wf.hit, wf.hitInst };
  RTC_CUDA(cudaMemsetAsync(cursor, 0, sizeof(uint32_t), ctx->stream));
  if (int rc = launch_k_trace<false, false, ExtendPathsAfter, true>(ctx, scene, p, 0u, count, cursor, nullptr)) return rc;
  return profile_end(ctx);
}

// Shadow rays of `queue` as closest-hit queries into hit[] / hitInst[] (after = past the ignored candidate already there).
int launch_connect_closest(rtc_context* ctx, const SceneDesc* scene, const WavefrontBuffers& wf, const uint32_t* queue, const uint32_t* count,
                           uint32_t* cursor, bool after)
{
  if (int rc = profile_begin(ctx, RTC_KERNEL_CONNECT)) return rc;
  RTC_CUDA(cudaMemsetAsync(cursor, 0, sizeof(uint32_t), ctx->stream));
  if (after)
  {
    ConnectClosest<true> p = { queue, wf.shadowOrg, wf.shadowDir, wf.hit, wf.hitInst };
    if (int rc = launch_k_trace<false, false, ConnectClosest<true>, true>(ctx, scene, p, 0u, count, cursor, nullptr)) return rc;
  }
  else
  {
    ConnectClosest<false> p = { queue, wf.shadowOrg, wf.shadowDir, wf.hit, wf.hitInst };
    if (int rc = launch_k_trace<false, false, ConnectClosest<false>, false>(ctx, scene, p, 0u, count, cursor, nullptr)) return rc;
  }
  return profile_end(ctx);
}

int read_stack_overflows(rtc_context* ctx, uint64_t* out)
{
  unsigned int v = 0;
  RTC_CUDA(cudaMemcpyFromSymbolAsync(&v, g_rtcStackOverflows, sizeof(v), 0, cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  uint64_t primary = 0;
  if (int rc = read_stack_overflows_primary(ctx, &primary)) return rc;
  *out = (uint64_t)v + primary;
  return 0;
}
