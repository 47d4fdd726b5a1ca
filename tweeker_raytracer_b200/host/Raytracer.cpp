#include "Raytracer.h"

#include <cstring>
#include <exception>
#include <iostream>
#include <string>
#include <thread>

#include "NcclComposite.h"

Raytracer::Raytracer(RendererStrategy strategy, const int interop, const unsigned int tex, const unsigned int pbo)
: m_strategy(strategy), m_interop(interop), m_tex(tex), m_pbo(pbo), m_isValid(false)
, m_visibleDevices(0), m_deviceOGL(-1), m_activeDevicesMask(0), m_iterationIndex(0), m_samplesPerPixel(1)
{
  RTC_CHECK(rtc_device_count(&m_visibleDevices));
  std::cout << "Raytracer() core version " << rtc_version() << ", " << m_visibleDevices << " visible CUDA device(s)" << std::endl;
}

Raytracer::~Raytracer()
{
  // Launches are asynchronous (render(count) enqueues without a sync) and the multi-GPU strategies share one frame: every
  // device must be idle before the first one is deleted and frees it.  Pending, never-observed iterations are dropped.
  m_pendingCount = 0;
  for (Device* device : m_activeDevices)
  {
    try { device->activateContext(); device->synchronizeStream(); } catch (std::exception const& e) { std::cerr << e.what() << std::endl; }
  }
  if (m_processGroup && !m_activeDevices.empty())
  {
    rtc_context* ctx = m_activeDevices[0]->getContext();
    RTC_CHECK_NO_THROW(rtc_synchronize(ctx));
    if (m_combined) RTC_CHECK_NO_THROW(rtc_free(ctx, m_combined));
    if (m_combinedHost) RTC_CHECK_NO_THROW(rtc_host_free(ctx, m_combinedHost));
  }
  ncclGroupDestroy(m_processGroup);
  for (Device* device : m_activeDevices) delete device;
}

void Raytracer::joinProcessGroup(const int rank, const int world, const char id[128])
{
  if (world < 1 || rank < 0 || world <= rank) throw std::runtime_error("ERROR: joinProcessGroup() rank/world out of range");
  if (m_activeDevices.size() != 1) throw std::runtime_error("ERROR: joinProcessGroup() needs exactly one active device per process (strategy 0)");
  if (m_processGroup) throw std::runtime_error("ERROR: joinProcessGroup() called twice");
  // The ranks' running averages are combined with an unweighted mean, which is only the mean of all samples while every
  // rank renders the same number of iterations: a sample count the ranks cannot share equally is refused, not truncated.
  if (m_samplesPerPixel % (unsigned int)world != 0u)
    throw std::runtime_error("ERROR: joinProcessGroup() samplesSqrt^2 = " + std::to_string(m_samplesPerPixel) + " is not divisible by the " + std::to_string(world) + " ranks");
  flush();
  m_processGroup = ncclProcessGroupJoin(rank, world, id, m_activeDevices[0]->m_ordinal);
  m_rank = rank;
  m_world = world;
  m_iterationIndex = 0;
  applySeedOffsets();
}

void Raytracer::reduceMeanToRoot(const uint64_t src, const uint64_t dst, const size_t count)
{
  if (!m_processGroup) throw std::runtime_error("ERROR: reduceMeanToRoot() without joinProcessGroup()");
  flush();
  ncclProcessGroupReduceMean(m_processGroup, src, dst, count, rtc_context_stream(m_activeDevices[0]->getContext()));
}

const void* Raytracer::getLocalOutputBufferHost()
{
  flush();
  return m_activeDevices.empty() ? nullptr : m_activeDevices[0]->getOutputBufferHost();
}

void Raytracer::applySeedOffsets()
{
  const unsigned int offset = (unsigned int)m_rank * getSamplesPerPixelLocal();
  for (Device* d : m_activeDevices) d->setSeedOffset(1 < m_world ? offset : 0u);
}

// Collective: mean of the ranks' running averages -> rank 0 (ncclReduce with ncclAvg on the render stream, so it is
// ordered behind the launches without a host synchronisation), then rank 0 reads the mean frame back.  The other ranks
// return nullptr: the frame lives on rank 0, and seven more 33 MB read-backs per step would only compete with rank 0's for
// host memory bandwidth (getLocalOutputBufferHost() fetches a rank's own running average when a tool wants it).
const void* Raytracer::combineProcessGroup()
{
  Device* device = m_activeDevices[0];
  rtc_context* ctx = device->getContext();
  SystemData const& sys = device->getSystemData();
  const size_t pixels = (size_t)sys.resolution.x * (size_t)sys.resolution.y;
  // A rank must never leave the collective to the others: a frame fetched before the first render() is the (zeroed) frame the
  // first render would allocate, not an exception on this rank while the other ranks wait in ncclReduce.
  if (device->getOutputBufferDevice() == 0) { void* buffer = nullptr; device->renderIterations(0, 0, &buffer); }
  if (device->getOutputBufferDevice() == 0) throw std::runtime_error("ERROR: getOutputBufferHost() could not allocate the frame");
  if (m_rank == 0 && m_combinedPixels != pixels)
  {
    RTC_CHECK(rtc_synchronize(ctx));
    if (m_combined) RTC_CHECK(rtc_free(ctx, m_combined));
    if (m_combinedHost) RTC_CHECK(rtc_host_free(ctx, m_combinedHost));
    RTC_CHECK(rtc_malloc(ctx, sizeof(float4) * pixels, &m_combined));
    RTC_CHECK(rtc_host_alloc(ctx, sizeof(float4) * pixels, &m_combinedHost));
    m_combinedPixels = pixels;
  }
  reduceMeanToRoot(device->getOutputBufferDevice(), m_combined, pixels * 4);
  if (m_rank != 0) return nullptr;
  RTC_CHECK(rtc_download(ctx, m_combinedHost, m_combined, sizeof(float4) * pixels));
  RTC_CHECK(rtc_synchronize(ctx));
  return m_combinedHost;
}

template <class DeviceType>
void Raytracer::createDevices(const int devicesMask, const int miss, const bool onlyFirst)
{
  std::vector<int> ordinals;
  for (int ordinal = 0; ordinal < m_visibleDevices && ordinal < 32; ++ordinal)
  {
    if (devicesMask & (1 << ordinal)) { ordinals.push_back(ordinal); if (onlyFirst) break; }
  }
  const int count = (int)ordinals.size();
  for (int index = 0; index < count; ++index)
  {
    const int ordinal = ordinals[index];
    m_activeDevices.push_back(new DeviceType(m_strategy, ordinal, index, count, miss, m_interop, m_tex, m_pbo));
    m_activeDevicesMask |= (1u << ordinal);
    char name[256] = "";
    RTC_CHECK(rtc_device_name(ordinal, name, (int)sizeof(name)));
    std::cout << "Raytracer() Using device " << ordinal << ": " << name << std::endl;
  }
  m_isValid = !m_activeDevices.empty();
}

// Peer-to-peer bit matrix and islands (Raytracer.cpp:109-234).  On an NVSwitch box all GPUs form one island.
bool Raytracer::enablePeerAccess()
{
  const size_t n = m_activeDevices.size();
  m_peerConnections.assign(n, 0u);
  for (size_t i = 0; i < n; ++i)
  {
    m_peerConnections[i] |= (1u << i);
    for (size_t j = 0; j < n; ++j)
    {
      if (i == j) continue;
      int can = 0;
      RTC_CHECK(rtc_peer_can_access(m_activeDevices[i]->m_ordinal, m_activeDevices[j]->m_ordinal, &can));
      if (can)
      {
        RTC_CHECK(rtc_peer_enable(m_activeDevices[i]->getContext(), m_activeDevices[j]->getContext()));
        m_peerConnections[i] |= (1u << j);
      }
    }
  }
  // islands: greedy grouping of devices which all see each other
  m_peerIslands.clear();
  std::vector<bool> placed(n, false);
  for (size_t i = 0; i < n; ++i)
  {
    if (placed[i]) continue;
    std::vector<int> island(1, (int)i);
    placed[i] = true;
    for (size_t j = i + 1; j < n; ++j)
    {
      if (placed[j]) continue;
      bool all = true;
      for (int k : island) all = all && (m_peerConnections[k] & (1u << j)) && (m_peerConnections[j] & (1u << k));
      if (all) { island.push_back((int)j); placed[j] = true; }
    }
    m_peerIslands.push_back(island);
  }
  return m_peerIslands.size() <= 1;
}

void Raytracer::disablePeerAccess()
{
  const size_t n = m_activeDevices.size();
  for (size_t i = 0; i < n && i < m_peerConnections.size(); ++i)
    for (size_t j = 0; j < n; ++j)
      if (i != j && (m_peerConnections[i] & (1u << j)))
        RTC_CHECK(rtc_peer_disable(m_activeDevices[i]->getContext(), m_activeDevices[j]->getContext()));
  m_peerConnections.clear();
  m_peerIslands.clear();
  for (size_t i = 0; i < n; ++i) m_peerIslands.push_back(std::vector<int>(1, (int)i));
}

void Raytracer::synchronize()
{
  flush();
  for (Device* device : m_activeDevices) { device->activateContext(); device->synchronizeStream(); }
}

void Raytracer::initTextures(std::map<std::string, EnvMap*> const& mapOfPictures) { for (Device* d : m_activeDevices) d->initTextures(mapOfPictures); }
void Raytracer::initCameras(std::vector<CameraDefinition> const& cameras) { for (Device* d : m_activeDevices) d->initCameras(cameras); }
void Raytracer::initLights(std::vector<LightDefinition> const& lights) { for (Device* d : m_activeDevices) d->initLights(lights); }
void Raytracer::initMaterials(std::vector<MaterialGUI> const& materialsGUI) { for (Device* d : m_activeDevices) d->initMaterials(materialsGUI); }
void Raytracer::initScene(std::shared_ptr<sg::Group> root, const unsigned int numGeometries) { for (Device* d : m_activeDevices) d->initScene(root, numGeometries); }

static unsigned int defaultCoalesceLimit(DeviceState const& state)
{
  const unsigned long long pixels = (unsigned long long)state.resolution.x * (unsigned long long)state.resolution.y;
  unsigned long long n = pixels ? (64ull << 20) / pixels : 1ull;      // the core keeps up to 64 Mi paths in flight per launch
  if (n < 1) n = 1;
  if (n > 64) n = 64;
  return (unsigned int)n;
}

void Raytracer::initState(DeviceState const& state)
{
  m_samplesPerPixel = (unsigned int)(state.samplesSqrt * state.samplesSqrt);
  if (!m_coalesceExplicit) m_coalesceLimit = defaultCoalesceLimit(state);
  for (Device* d : m_activeDevices) d->setState(state);
  applySeedOffsets();
}

// Every update restarts the accumulation (Raytracer.cpp:331-367).
void Raytracer::updateCamera(const int idCamera, CameraDefinition const& camera) { flush(); for (Device* d : m_activeDevices) d->updateCamera(idCamera, camera); m_iterationIndex = 0; }
void Raytracer::updateLight(const int idLight, LightDefinition const& light) { flush(); for (Device* d : m_activeDevices) d->updateLight(idLight, light); m_iterationIndex = 0; }
void Raytracer::updateMaterial(const int idMaterial, MaterialGUI const& src) { flush(); for (Device* d : m_activeDevices) d->updateMaterial(idMaterial, src); m_iterationIndex = 0; }
void Raytracer::updateInstanceTransforms(const unsigned int first, const unsigned int count, const float* matrices)
{
  flush();
  for (Device* d : m_activeDevices) d->updateInstanceTransforms(first, count, matrices);
  m_iterationIndex = 0;
}
// A new topology over the same instance boxes: hits, and so frames, do not change, and the accumulation goes on.
void Raytracer::rebuildInstanceLevel()
{
  flush();
  for (Device* d : m_activeDevices) d->rebuildInstanceLevel();
}
// A deformed mesh (an extension of the reference's Raytracer surface): refitted, or rebuilt after large deformation.
void Raytracer::updateGeometry(const unsigned int id, const TriangleAttributes* attributes, const size_t numAttributes, const bool rebuild)
{
  flush();
  for (Device* d : m_activeDevices) d->updateGeometry(id, attributes, numAttributes, rebuild);
  m_iterationIndex = 0;
}
void Raytracer::updateState(DeviceState const& state)
{
  // a new resolution makes the owner free and reallocate the shared frame: no device may still be writing to the old one
  synchronize();
  if (!m_coalesceExplicit) m_coalesceLimit = defaultCoalesceLimit(state);
  m_samplesPerPixel = (unsigned int)(state.samplesSqrt * state.samplesSqrt);
  for (Device* d : m_activeDevices) d->setState(state);
  applySeedOffsets();
  m_iterationIndex = 0;
}

unsigned int Raytracer::render(const unsigned int count) { return renderAll(count); }

// render(): count the iterations; enqueue them as one batch once the coalescing limit is reached (see Raytracer.h).
unsigned int Raytracer::renderAll(const unsigned int count)
{
  const unsigned int budget = getSamplesPerPixelLocal();    // == m_samplesPerPixel unless this process is one rank of several
  if (m_iterationIndex < budget)
  {
    unsigned int n = budget - m_iterationIndex;
    if (count < n) n = count;
    if (m_pendingCount == 0) m_pendingFirst = m_iterationIndex;
    m_pendingCount += n;
    m_iterationIndex += n;
    if (m_coalesceLimit <= m_pendingCount) flush();
  }
  return m_iterationIndex;
}

// All devices work on the same iteration indices.  The first device called allocates the shared buffers (the `void**
// buffer` protocol of Device::render, DeviceMultiGPUPeerAccess.cpp:110-125), so it is driven first; the others only enqueue
// kernels on their own streams and are driven by one host thread each -- with 8 GPUs a single thread issuing ~2000 launches
// per device and batch was what bounded the tile partition at 4K (profiles/c5_4k_r1.md).
void Raytracer::flush()
{
  if (m_pendingCount == 0) return;
  const unsigned int first = m_pendingFirst, n = m_pendingCount;
  m_pendingCount = 0;
  void* buffer = nullptr;
  if (m_activeDevices.empty()) return;
  m_activeDevices[0]->renderIterations(first, n, &buffer);
  const size_t others = m_activeDevices.size() - 1;
  if (others == 1) m_activeDevices[1]->renderIterations(first, n, &buffer);
  else if (1 < others)
  {
    std::vector<std::thread> workers;
    std::vector<std::exception_ptr> errors(others);
    for (size_t i = 0; i < others; ++i)
      workers.emplace_back([this, i, first, n, buffer, &errors]() {
        void* shared = buffer;
        try { m_activeDevices[i + 1]->renderIterations(first, n, &shared); } catch (...) { errors[i] = std::current_exception(); }
      });
    for (std::thread& t : workers) t.join();
    for (std::exception_ptr& e : errors) if (e) std::rethrow_exception(e);
  }
}

void Raytracer::getStats(rtc_stats& total)
{
  flush();
  std::memset(&total, 0, sizeof(total));
  for (Device* device : m_activeDevices)
  {
    rtc_stats s; device->getStats(s);
    total.radianceRays += s.radianceRays; total.shadowRays += s.shadowRays; total.pathSamples += s.pathSamples;
    total.kernelLaunches += s.kernelLaunches; total.lastTraceMs = s.lastTraceMs; total.stackOverflows += s.stackOverflows;
    total.cutoutGraphBuilds += s.cutoutGraphBuilds;
  }
}

// ---------------------------------------------------------------------------------------------------------------
RaytracerSingleGPU::RaytracerSingleGPU(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo)
: Raytracer(RS_INTERACTIVE_SINGLE_GPU, interop, tex, pbo)
{
  createDevices<DeviceSingleGPU>(devicesMask, miss, true);
}

RaytracerMultiGPUZeroCopy::RaytracerMultiGPUZeroCopy(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo)
: Raytracer(RS_INTERACTIVE_MULTI_GPU_ZERO_COPY, interop, tex, pbo)
{
  createDevices<DeviceMultiGPUZeroCopy>(devicesMask, miss, false);
}

const void* RaytracerMultiGPUZeroCopy::getOutputBufferHost()
{
  synchronize();
  return m_activeDevices[0]->getOutputBufferHost();
}

RaytracerMultiGPUPeerAccess::RaytracerMultiGPUPeerAccess(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo)
: Raytracer(RS_INTERACTIVE_MULTI_GPU_PEER_ACCESS, interop, tex, pbo)
{
  createDevices<DeviceMultiGPUPeerAccess>(devicesMask, miss, false);
  // the shared frame lives on one device: every active device must reach it (RaytracerMultiGPUPeerAccess.cpp:79-84)
  if (m_isValid && !enablePeerAccess())
  {
    std::cerr << "ERROR: RaytracerMultiGPUPeerAccess() the active devices do not form one peer-to-peer island." << std::endl;
    m_isValid = false;
  }
}

RaytracerMultiGPUPeerAccess::~RaytracerMultiGPUPeerAccess()
{
  m_pendingCount = 0;      // never-observed iterations are dropped
  try { synchronize(); disablePeerAccess(); } catch (std::exception const& e) { std::cerr << e.what() << std::endl; }
}

const void* RaytracerMultiGPUPeerAccess::getOutputBufferHost()
{
  synchronize();
  return m_activeDevices[0]->getOutputBufferHost();
}

// ---------------------------------------------------------------------------------------------------------------
struct RaytracerMultiGPULocalCopy::NcclState
{
  NcclGroup* group = nullptr;
  std::vector<uint64_t> scatter;   // per device: full-resolution frame holding only that device's pixels
  size_t pixels = 0;
};

RaytracerMultiGPULocalCopy::RaytracerMultiGPULocalCopy(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo)
: Raytracer(RS_INTERACTIVE_MULTI_GPU_LOCAL_COPY, interop, tex, pbo)
{
  createDevices<DeviceMultiGPULocalCopy>(devicesMask, miss, false);
  if (m_isValid) enablePeerAccess();   // peer copies fall back to staging through the host when this is not one island
}

RaytracerMultiGPULocalCopy::~RaytracerMultiGPULocalCopy()
{
  m_pendingCount = 0;      // never-observed iterations are dropped
  try
  {
    synchronize();
    if (m_nccl)
    {
      for (size_t i = 0; i < m_nccl->scatter.size(); ++i) if (m_nccl->scatter[i]) RTC_CHECK_NO_THROW(rtc_free(m_activeDevices[i]->getContext(), m_nccl->scatter[i]));
      ncclGroupDestroy(m_nccl->group);
      delete m_nccl;
    }
    disablePeerAccess();
  }
  catch (std::exception const& e) { std::cerr << e.what() << std::endl; }
}

// The reference composites device 0 twice when no OpenGL device exists (RaytracerMultiGPULocalCopy.cpp:141-147);
// the result is the same, so each device is composited once here.
void RaytracerMultiGPULocalCopy::composite()
{
  flush();
  if (m_compositeMode == COMPOSITE_NCCL_REDUCE && 1 < m_activeDevices.size()) { compositeNccl(); return; }
  synchronize();
  for (Device* device : m_activeDevices) m_activeDevices[0]->compositor(device);
}

// Every device scatters its own texel slab into a zeroed full-resolution frame (pixel ownership is disjoint), then
// ONE ncclReduce(sum) over NVLink lands the complete frame on device 0: x + 0 + ... + 0 is exact, so the result is
// bit-identical to the serial peer-copy compositor.
void RaytracerMultiGPULocalCopy::compositeNccl()
{
  const size_t n = m_activeDevices.size();
  DeviceMultiGPULocalCopy* root = static_cast<DeviceMultiGPULocalCopy*>(m_activeDevices[0]);
  SystemData const& sys = root->getSystemData();
  const size_t pixels = (size_t)sys.resolution.x * (size_t)sys.resolution.y;
  if (!m_nccl)
  {
    m_nccl = new NcclState();
    std::vector<int> ordinals;
    for (Device* d : m_activeDevices) ordinals.push_back(d->m_ordinal);
    m_nccl->group = ncclGroupCreate((int)n, ordinals.data());
    m_nccl->scatter.assign(n, 0);
  }
  if (m_nccl->pixels != pixels)
  {
    for (size_t i = 0; i < n; ++i)
    {
      if (m_nccl->scatter[i]) RTC_CHECK(rtc_free(m_activeDevices[i]->getContext(), m_nccl->scatter[i]));
      RTC_CHECK(rtc_malloc(m_activeDevices[i]->getContext(), sizeof(float4) * pixels, &m_nccl->scatter[i]));
    }
    m_nccl->pixels = pixels;
  }
  for (size_t i = 0; i < n; ++i)
  {
    DeviceMultiGPULocalCopy* d = static_cast<DeviceMultiGPULocalCopy*>(m_activeDevices[i]);
    RTC_CHECK(rtc_memset(d->getContext(), m_nccl->scatter[i], 0, sizeof(float4) * pixels));
    CompositorData args;
    args.outputBuffer = m_nccl->scatter[i];
    args.tileBuffer = d->getTexelBuffer();
    args.resolution = sys.resolution; args.tileSize = sys.tileSize; args.tileShift = sys.tileShift;
    args.launchWidth = d->getLaunchWidth(); args.deviceCount = (int)n; args.deviceIndex = d->m_index;
    RTC_CHECK(rtc_composite(d->getContext(), &args));
  }
  std::vector<uint64_t> streams(n);
  for (size_t i = 0; i < n; ++i) streams[i] = rtc_context_stream(m_activeDevices[i]->getContext());
  ncclGroupReduceSum(m_nccl->group, m_nccl->scatter.data(), root->getOutputBuffer(), pixels * 4, streams.data());
  synchronize();
}

const void* RaytracerMultiGPULocalCopy::getOutputBufferHost()
{
  composite();
  return m_activeDevices[0]->getOutputBufferHost();
}
