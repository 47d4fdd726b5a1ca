// tests/native/device_trace_host.cpp -- TEST INFRASTRUCTURE: the device-side queries of include/rtc_device.cuh compiled for the
// host.  tests/native/trace_host.cpp is included unchanged (the intrinsics with their IEEE meaning, the host scene); one host thread
// plays one calling thread.  The scene's node, leaf, instance-record, triangle and mask fetches of the traversal all go through
// __ldg: the overloads below count them (exact non-template matches, so they win over trace_host.cpp's template).
#include <cstdint>

#include <cuda_runtime.h>

static uint64_t g_sceneReads = 0;
static inline uint4 __ldg(const uint4* p) { ++g_sceneReads; return *p; }
static inline float4 __ldg(const float4* p) { ++g_sceneReads; return *p; }
static inline uint32_t __ldg(const uint32_t* p) { ++g_sceneReads; return *p; }
static inline uint8_t __ldg(const uint8_t* p) { ++g_sceneReads; return *p; }

#include "trace_host.cpp"
#include "rtc_device.cuh"

extern "C" {

// The scene as the library lays it out behind topObject: the SceneDesc, then the SceneDeviceRecord {instMasks, usable, abi}.
// rayMasks / rayFlags: per ray.  any: 0 closest (hits), 1 any (occluded).  status: per ray.  reads: the scene fetches of the
// whole call.
int dth_trace(const th_scene* ws, uint32_t numTlasNodes, uint32_t numTlasLeaves, uint32_t numGas, const uint32_t* numGasNodes,
              const uint32_t* numGasTris, const uint8_t* instMasks, uint32_t usable, uint32_t abi, const rtc_ray* rays, uint64_t n,
              const uint32_t* rayMasks, const uint32_t* rayFlags, int any, rtc_hit* hits, uint32_t* occluded, int* status, uint64_t* reads)
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
  for (uint64_t i = 0; i < n; ++i)
  {
    if (any) status[i] = rtc_device_trace_any(topObject, rays[i], occluded + i, rayMasks[i], rayFlags[i]);
    else     status[i] = rtc_device_trace_closest(topObject, rays[i], hits + i, rayMasks[i], rayFlags[i]);
  }
  *reads = g_sceneReads;
  return 0;
}

// the header's constants, so the tests need not restate them
void dth_constants(int out[5])
{
  out[0] = RTC_DEVICE_OK; out[1] = RTC_DEVICE_SCENE_UNUSABLE; out[2] = RTC_DEVICE_BAD_ARGUMENT; out[3] = RTC_DEVICE_ABI_MISMATCH;
  out[4] = (int)kSceneDeviceAbi;
}

} // extern "C"
