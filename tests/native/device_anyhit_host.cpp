// tests/native/device_anyhit_host.cpp -- TEST INFRASTRUCTURE: the any-hit queries of include/rtc_device.cuh compiled for the host
// over an exported wide BVH, as tests/native/device_trace_host.cpp does for the plain queries (trace_host.cpp included unchanged,
// the scene's fetches counted through __ldg).  One host thread plays one calling thread; its callback is a lambda that decides
// with anyhit_predicates.h and records every call.
#include <cstdint>
#include <set>
#include <utility>

#include <cuda_runtime.h>

static uint64_t g_sceneReads = 0;
static inline uint4 __ldg(const uint4* p) { ++g_sceneReads; return *p; }
static inline float4 __ldg(const float4* p) { ++g_sceneReads; return *p; }
static inline uint32_t __ldg(const uint32_t* p) { ++g_sceneReads; return *p; }
static inline uint8_t __ldg(const uint8_t* p) { ++g_sceneReads; return *p; }

#include "trace_host.cpp"
#include "rtc_device.cuh"
#include "anyhit_predicates.h"

extern "C" {

// The scene laid out behind topObject as the library lays it out (see dth_trace).  Per ray: rayMasks, rayFlags, the predicate's
// parameters p0 / p1.  mode: 0 closest_anyhit (hits), 1 any_anyhit (occluded), 2 plain closest, 3 plain any.  end: accepts are
// RTC_ANYHIT_ACCEPT_AND_END.  Calls of ray i: calls[i] (the first k recorded in records[i * k ...]), digest[3 i ...] (count, sum,
// XOR of anyhit_predicates.h), and *duplicates counts calls on an (instance, primitive) the ray had already offered.
int dah_trace(const th_scene* ws, uint32_t numTlasNodes, uint32_t numTlasLeaves, uint32_t numGas, const uint32_t* numGasNodes,
              const uint32_t* numGasTris, const uint8_t* instMasks, uint32_t usable, uint32_t abi, const rtc_ray* rays, uint64_t n,
              const uint32_t* rayMasks, const uint32_t* rayFlags, int mode, int pred, const uint32_t* p0, const uint32_t* p1, int end,
              uint32_t k, rtc_hit* hits, uint32_t* occluded, int* status, uint32_t* calls, ahp_record* records, uint32_t* digest,
              uint64_t* duplicates, uint64_t* reads)
{
  HostScene hs;
  build_host_scene(hs, ws, numTlasNodes, numTlasLeaves, numGas, numGasNodes, numGasTris);
  uint8_t* top = static_cast<uint8_t*>(hs.aligned(kSceneDeviceRecordOffset + sizeof(SceneDeviceRecord)));
  std::memcpy(top, &hs.sc, sizeof(SceneDesc));
  SceneDeviceRecord rec;
  rec.instMasks = static_cast<const uint8_t*>(hs.copy(instMasks, ws->numInstances));
  rec.usable = usable; rec.abi = abi;
  std::memcpy(top + kSceneDeviceRecordOffset, &rec, sizeof(rec));
  const uint64_t topObject = (uint64_t)(uintptr_t)top;

  g_sceneReads = 0;
  *duplicates = 0;
  for (uint64_t i = 0; i < n; ++i)
  {
    uint32_t count = 0, d[3] = { 0u, 0u, 0u };
    std::set<std::pair<uint32_t, uint32_t>> seen;
    auto anyHit = [&](const rtc_candidate& c) {
      if (count < k) std::memcpy(records + i * k + count, &c, sizeof(ahp_record));
      ++count;
      ahp_digest_add(d, c.t, c.u, c.v, c.inst, c.prim, c.frontFacing);
      if (!seen.insert(std::make_pair(c.inst, c.prim)).second) ++*duplicates;
      return ahp_decide(pred, c.t, c.u, c.v, c.inst, c.prim, c.frontFacing, p0[i], p1[i], end);
    };
    switch (mode)
    {
    case 0: status[i] = rtc_device_trace_closest_anyhit(topObject, rays[i], hits + i, anyHit, rayMasks[i], rayFlags[i]); break;
    case 1: status[i] = rtc_device_trace_any_anyhit(topObject, rays[i], occluded + i, anyHit, rayMasks[i], rayFlags[i]); break;
    case 2: status[i] = rtc_device_trace_closest(topObject, rays[i], hits + i, rayMasks[i], rayFlags[i]); break;
    default: status[i] = rtc_device_trace_any(topObject, rays[i], occluded + i, rayMasks[i], rayFlags[i]); break;
    }
    calls[i] = count;
    digest[3 * i] = d[0]; digest[3 * i + 1] = d[1]; digest[3 * i + 2] = d[2];
  }
  *reads = g_sceneReads;
  return 0;
}

// the header's constants, so the tests need not restate them
void dah_constants(int out[4])
{
  out[0] = RTC_ANYHIT_IGNORE; out[1] = RTC_ANYHIT_ACCEPT; out[2] = RTC_ANYHIT_ACCEPT_AND_END; out[3] = (int)sizeof(rtc_candidate);
}

} // extern "C"
