// rtc_device.cuh -- ray queries from the caller's own CUDA kernels: the device-side counterpart of optixTrace.
//
//   __global__ void my_kernel(uint64_t topObject, ...)
//   {
//     rtc_ray ray = ...;                                    // origin, tmin, direction, tmax
//     rtc_hit hit;
//     if (rtc_device_trace_closest(topObject, ray, &hit) == RTC_DEVICE_OK && hit.inst != 0xffffffffu) ...
//   }
//
// topObject is the handle rtc_ias_build / rtc_ias_create return (SystemData::topObject).  Compile the kernel with
// -I<repository>/include as its only include path (INTEGRATION.md, "Tracing from your own kernels").  Detect the feature by this
// header: rtc_version() is unchanged.
//
// Results.  For every ray, mask and flag set the result equals rtc_trace_closest_ex / rtc_trace_any_ex with the same mask and
// flags, bit for bit: t, u, v, inst, prim and occluded.  The calls run the library's own traversal (tweeker_raytracer_b200/csrc/
// trace.cuh), always its filtered variant: visibilityMask and rayFlags (RTC_RAY_CULL_*) are ordinary arguments, so every ray may
// have its own, and with (0xFF, 0) an instance of mask 0 is never entered, exactly as in the _ex calls.
//
// Status.  RTC_DEVICE_OK, or:
//   RTC_DEVICE_BAD_ARGUMENT    visibilityMask > 0xFF or a rayFlags bit other than RTC_RAY_CULL_*;
//   RTC_DEVICE_SCENE_UNUSABLE  the scene is one rtc_trace_* would refuse at this point of the context stream: a GAS it instances
//                              was refitted, rebuilt or built again (rtc_gas_refit / _rebuild / _build_device; for a scene of
//                              rtc_ias_create any GAS of the context) and the scene has not been updated since, or was destroyed;
//   RTC_DEVICE_ABI_MISMATCH    the scene was made by a library built from another version of this header.
// Every status but RTC_DEVICE_OK writes a miss (t = -1, u = v = 0, inst = prim = 0xffffffff; occluded = 0) and reads no node,
// leaf or instance record of the scene.
//
// Contract.
//   - The query reads the scene when the kernel runs, not when it is launched.  Order the kernel after the library calls it must
//     see (builds, updates, rebuilds, rtc_scene_set_instance_masks) by launching it on rtc_context_stream(ctx), or with events;
//     order the library calls that follow it the same way.
//   - Call it on the context's device only.  Scenes of a peer GPU are not supported.
//   - A destroyed scene (rtc_scene_destroy) is a freed buffer: its topObject must not be passed any more.
//   - Any kernel, block size, divergent branch or partial warp: the calls use no warp collective, no shared memory and no
//     __syncthreads.  Each call keeps its traversal stack (8 + 32 entries, 320 B) in local memory.
//   - Rays whose traversal stack overflows are counted in rtc_device_stack_overflows, a __device__ variable of the calling
//     translation unit, not in rtc_stats.  It is never non-zero for the trees this library builds.
//   - Compiler flags: the results are bit-identical under nvcc's defaults and under -fmad=false (the triangle test pins its
//     rounding with intrinsics; only the conservative box test may contract).  -ftz=true and --use_fast_math flush the
//     intersector's denormals and are outside this contract; nvcc defines no macro the header could test for them.
//   - Several translation units of one -rdc=true program may include this header: every definition in it is local to its unit.
//
// Any-hit callbacks (the any-hit program of OptiX: optixIgnoreIntersection, optixTerminateRay).
//   rtc_device_trace_closest_anyhit / rtc_device_trace_any_anyhit take the caller's code as `anyHit`: anything callable as
//   anyHit(const rtc_candidate&) whose result converts to int, usually a plain lambda written in the kernel,
//     [&](const rtc_candidate& c) { return alpha(c.inst, c.prim, c.u, c.v) > 0.5f; }
//   (no __device__ on it and no --extended-lambda: a lambda inside device code is a device lambda).  It returns
//   RTC_ANYHIT_IGNORE (0), RTC_ANYHIT_ACCEPT_AND_END (2) or anything else, which accepts; a bool predicate reads as it is written.
//   - When it runs: only on a candidate of an instance the ray's mask enters, that passes the watertight test and the cull flags,
//     with t > tmin, and that would become the result: for the closest query it beats the best hit so far (t < tmax, or smaller
//     in (t, instance, primitive) than the hit accepted so far), for the any query t < tmax.  Never on a refused call, nor on an
//     empty interval.
//   - At most once per (instance, primitive) and ray: every triangle has one leaf slot and every instance one instance-level leaf.
//   - Ignore leaves the query as it was.  Accept in the closest query makes the candidate the best hit and shrinks tmax to its t;
//     in the any query it ends the query with *occluded = 1.  Accept-and-end makes the candidate the result and ends the query.
//   - Reproducible: (a) when the decision is a pure function of the candidate's fields and never accept-and-end, the closest query
//     returns the smallest accepted candidate in (t, instance, primitive) order -- brute force over all triangles with the same
//     predicate, whatever the tree.  (b) An any query whose callback always ignores calls it exactly once for every candidate
//     of the ray after masks, culling and (tmin, tmax).  (c) A callback that always accepts returns what rtc_device_trace_closest
//     / _any return, bit for bit.  The order of the calls, their number in the closest query, and the result of accept-and-end or
//     of a stateful decision (including floating-point reductions such as a transmittance product) depend on the node order of
//     the tree: deterministic for one structure, but not part of this contract.
//   - The callback may read and write any memory the kernel can.  It must not call rtc_device_trace_* (nested queries are not
//     supported).  Every other rule above holds unchanged.
#pragma once

#ifndef RTC_STACK_OVERFLOW_COUNTER
#define RTC_STACK_OVERFLOW_COUNTER rtc_device_stack_overflows
#define RTC_STACK_OVERFLOW_STORAGE static
#endif
#include "../tweeker_raytracer_b200/csrc/trace.cuh"

// status of a device-side query
enum { RTC_DEVICE_OK = 0, RTC_DEVICE_SCENE_UNUSABLE = 1, RTC_DEVICE_BAD_ARGUMENT = 2, RTC_DEVICE_ABI_MISMATCH = 3 };

// One candidate intersection, as an any-hit callback sees it.  t, inst, prim as in rtc_hit; u, v are the barycentrics the closest
// query returns for it (same operands, same bits); frontFacing: 1 when the candidate is front-facing in object space (the rule
// of RTC_RAY_CULL_*), else 0.
struct rtc_candidate
{
  float    t, u, v;
  uint32_t inst, prim;
  uint32_t frontFacing;
};

// decision of an any-hit callback; any other value counts as RTC_ANYHIT_ACCEPT (so a bool predicate reads as "accept")
enum { RTC_ANYHIT_IGNORE = 0, RTC_ANYHIT_ACCEPT = 1, RTC_ANYHIT_ACCEPT_AND_END = 2 };

// The traversal offers a candidate's raw operands (trace.cuh Traversal, ANYHIT); this builds the rtc_candidate from them.
template <class F>
struct rtc_device_anyhit_adapter
{
  F& f;
  __device__ __forceinline__ int operator()(float t, float det, float V, float W, uint32_t inst, uint32_t prim) const
  {
    rtc_candidate c;
    c.t = t; c.u = __fdiv_rn(V, det); c.v = __fdiv_rn(W, det); c.inst = inst; c.prim = prim; c.frontFacing = det > 0.0f ? 1u : 0u;
    return static_cast<int>(f(static_cast<const rtc_candidate&>(c)));
  }
};

// One ray through the filtered traversal, one thread on its own: the stack and the ray words that the batch kernels keep in
// shared memory (trace.cuh Traversal) are per-thread arrays here (BLOCK = 1), and the triangle tests of a step are not capped.
// ANYHIT: TraceNoAnyHit (anyHit null) or an rtc_device_anyhit_adapter.
template <bool ANY, class ANYHIT = TraceNoAnyHit>
static __device__ __forceinline__ int rtc_device_trace_impl(uint64_t topObject, const rtc_ray& ray, uint32_t visibilityMask, uint32_t rayFlags,
                                                            TraceHit& h, ANYHIT* anyHit = nullptr)
{
  h.t = -1.0f; h.u = 0.0f; h.v = 0.0f; h.inst = 0xffffffffu; h.prim = 0xffffffffu;
  if (visibilityMask > 0xFFu || (rayFlags & ~(RTC_RAY_CULL_BACK_FACING | RTC_RAY_CULL_FRONT_FACING))) return RTC_DEVICE_BAD_ARGUMENT;
  const SceneDeviceRecord rec = *reinterpret_cast<const SceneDeviceRecord*>((uintptr_t)(topObject + kSceneDeviceRecordOffset));
  if (rec.abi != kSceneDeviceAbi) return RTC_DEVICE_ABI_MISMATCH;
  if (!rec.usable) return RTC_DEVICE_SCENE_UNUSABLE;
  const SceneDesc sc = *reinterpret_cast<const SceneDesc*>((uintptr_t)topObject);
  Traversal<ANY, false, 1, false, 0, true, ANYHIT> tr;
  uint2 smStack[RTC_SM_STACK], lmStack[RTC_LM_STACK];
  float smRay[RTC_SM_RAY_WORDS];
  tr.smStack = smStack; tr.lmStack = lmStack; tr.smRay = smRay;
  TraceFilter filt;
  filt.masks = rec.instMasks; filt.rayMask = visibilityMask; filt.cullFlags = rayFlags;
  if (tr.begin(sc, make_float4(ray.ox, ray.oy, ray.oz, ray.tmin), make_float4(ray.dx, ray.dy, ray.dz, ray.tmax)))
    while (tr.step(sc, filt, anyHit)) {}
  h = tr.result();
  return RTC_DEVICE_OK;
}

// Closest hit in (tmin, tmax): smallest t, ties to the smaller (instance, primitive).  Miss: t = -1, inst = prim = 0xffffffff.
static __device__ __forceinline__ int rtc_device_trace_closest(uint64_t topObject, const rtc_ray& ray, rtc_hit* hit,
                                                               uint32_t visibilityMask = 0xFFu, uint32_t rayFlags = 0u)
{
  TraceHit h;
  const int status = rtc_device_trace_impl<false>(topObject, ray, visibilityMask, rayFlags, h);
  hit->t = h.t; hit->u = h.u; hit->v = h.v; hit->inst = h.inst; hit->prim = h.prim;
  return status;
}

// Any hit in (tmin, tmax): *occluded = 1 when there is one, else 0.
static __device__ __forceinline__ int rtc_device_trace_any(uint64_t topObject, const rtc_ray& ray, uint32_t* occluded,
                                                           uint32_t visibilityMask = 0xFFu, uint32_t rayFlags = 0u)
{
  TraceHit h;
  const int status = rtc_device_trace_impl<true>(topObject, ray, visibilityMask, rayFlags, h);
  *occluded = h.inst != 0xffffffffu ? 1u : 0u;
  return status;
}

// Closest hit with the caller's any-hit code: the smallest candidate in (t, instance, primitive) order that anyHit accepts, or the
// one it accepts and ends with.  anyHit(const rtc_candidate&) -> int or bool; see "Any-hit callbacks" above.
template <class AnyHit>
static __device__ __forceinline__ int rtc_device_trace_closest_anyhit(uint64_t topObject, const rtc_ray& ray, rtc_hit* hit, AnyHit&& anyHit,
                                                                      uint32_t visibilityMask = 0xFFu, uint32_t rayFlags = 0u)
{
  using F = typename std::remove_reference<AnyHit>::type;
  rtc_device_anyhit_adapter<F> adapter{anyHit};
  TraceHit h;
  const int status = rtc_device_trace_impl<false>(topObject, ray, visibilityMask, rayFlags, h, &adapter);
  hit->t = h.t; hit->u = h.u; hit->v = h.v; hit->inst = h.inst; hit->prim = h.prim;
  return status;
}

// Any hit with the caller's any-hit code: *occluded = 1 at the first candidate anyHit accepts, else 0.
template <class AnyHit>
static __device__ __forceinline__ int rtc_device_trace_any_anyhit(uint64_t topObject, const rtc_ray& ray, uint32_t* occluded, AnyHit&& anyHit,
                                                                  uint32_t visibilityMask = 0xFFu, uint32_t rayFlags = 0u)
{
  using F = typename std::remove_reference<AnyHit>::type;
  rtc_device_anyhit_adapter<F> adapter{anyHit};
  TraceHit h;
  const int status = rtc_device_trace_impl<true>(topObject, ray, visibilityMask, rayFlags, h, &adapter);
  *occluded = h.inst != 0xffffffffu ? 1u : 0u;
  return status;
}
