// tests/native/trace_host_ex.cpp -- TEST INFRASTRUCTURE: the FILTER traversal of csrc/trace.cuh (rtc_trace_*_ex: instance
// visibility masks and face culling) compiled for the host.  tests/native/trace_host.cpp is included unchanged: the same
// intrinsics with their IEEE meaning and the same host scene; one host thread plays one lane.
#include "trace_host.cpp"

extern "C" {

// masks: one byte per instance; rayMask; cullFlags: RTC_RAY_CULL_*; cap: the TRICAP schedule (0, 1 or 2) the timed kernels
// instantiate.  Otherwise as th_trace without skip keys (the IEEE reciprocal of the counting kernels).
int th_trace_ex(const th_scene* ws, uint32_t numTlasNodes, uint32_t numTlasLeaves, uint32_t numGas, const uint32_t* numGasNodes,
                const uint32_t* numGasTris, const rtc_ray* rays, uint64_t n, int any, const uint8_t* masks, uint32_t rayMask,
                uint32_t cullFlags, int cap, rtc_hit* hits, uint64_t counts[3], uint64_t* stackOverflows)
{
  HostScene hs;
  build_host_scene(hs, ws, numTlasNodes, numTlasLeaves, numGas, numGasNodes, numGasTris);
  const SceneDesc& sc = hs.sc;
  TraceFilter filt;
  filt.masks = (const uint8_t*)hs.copy(masks, ws->numInstances);
  filt.rayMask = rayMask; filt.cullFlags = cullFlags;

  counts[0] = counts[1] = counts[2] = 0;
  const unsigned overflowsBefore = RTC_STACK_OVERFLOW_COUNTER;
  uint2 smStack[RTC_SM_STACK]; float smRay[RTC_SM_RAY_WORDS]; uint2 lmStack[RTC_LM_STACK];
  auto run = [&](auto& tr, const rtc_ray& r) {
    tr.smStack = smStack; tr.smRay = smRay; tr.lmStack = lmStack;
    if (tr.begin(sc, make_float4(r.ox, r.oy, r.oz, r.tmin), make_float4(r.dx, r.dy, r.dz, r.tmax)))
    {
      while (tr.step(sc, filt)) {}
      counts[0] += tr.counts.nodes; counts[1] += tr.counts.tris; counts[2] += tr.counts.insts;
    }
    return tr.result();
  };
  for (uint64_t i = 0; i < n; ++i)
  {
    TraceHit h;
    if (any)
    {
      if (cap == 1)      { Traversal<true, true, 1, false, 1, true> tr; h = run(tr, rays[i]); }
      else if (cap == 2) { Traversal<true, true, 1, false, 2, true> tr; h = run(tr, rays[i]); }
      else               { Traversal<true, true, 1, false, 0, true> tr; h = run(tr, rays[i]); }
    }
    else
    {
      if (cap == 1)      { Traversal<false, true, 1, false, 1, true> tr; h = run(tr, rays[i]); }
      else if (cap == 2) { Traversal<false, true, 1, false, 2, true> tr; h = run(tr, rays[i]); }
      else               { Traversal<false, true, 1, false, 0, true> tr; h = run(tr, rays[i]); }
    }
    if (hits) { hits[i].t = h.t; hits[i].u = h.u; hits[i].v = h.v; hits[i].inst = h.inst; hits[i].prim = h.prim; }
  }
  if (stackOverflows) *stackOverflows = RTC_STACK_OVERFLOW_COUNTER - overflowsBefore;
  return 0;
}

} // extern "C"
