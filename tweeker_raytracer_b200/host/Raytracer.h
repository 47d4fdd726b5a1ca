// Raytracer.h -- the strategy layer of rtigo3 (apps/rtigo3/inc/Raytracer.h:49-101 and the four derived
// classes).  A Raytracer owns the active Devices (bits of devicesMask that exist), broadcasts init*/update*
// to them, advances the iteration counter in render() and produces the final float4 frame.
//   RaytracerSingleGPU            RaytracerSingleGPU.cpp:38-92
//   RaytracerMultiGPUZeroCopy     RaytracerMultiGPUZeroCopy.cpp:38-129
//   RaytracerMultiGPUPeerAccess   RaytracerMultiGPUPeerAccess.cpp:38-160
//   RaytracerMultiGPULocalCopy    RaytracerMultiGPULocalCopy.cpp:38-173
// B200 additions: render(count) enqueues several iterations at once, and the local-copy strategy can combine
// the per-GPU results with one NCCL reduce over NVLink instead of N serial peer copies (setCompositeMode).
// One process per GPU (torchrun-style): joinProcessGroup(rank, world, id) turns a single-GPU Raytracer into rank `rank`
// of a sample-range partition -- it renders the iterations [rank * spp/world, (rank+1) * spp/world) as its own
// running average, and getOutputBufferHost() becomes a collective that lands the mean of the ranks' frames on rank 0
// with one ncclReduce over NVLink (the other ranks get nullptr).
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "Devices.h"

class Raytracer
{
public:
  Raytracer(RendererStrategy strategy, const int interop, const unsigned int tex, const unsigned int pbo);
  virtual ~Raytracer();

  bool enablePeerAccess();    // fills m_peerConnections and m_peerIslands; false when more than one island exists
  void disablePeerAccess();
  void synchronize();

  virtual void initTextures(std::map<std::string, EnvMap*> const& mapOfPictures);
  virtual void initCameras(std::vector<CameraDefinition> const& cameras);
  virtual void initLights(std::vector<LightDefinition> const& lights);
  virtual void initMaterials(std::vector<MaterialGUI> const& materialsGUI);
  virtual void initScene(std::shared_ptr<sg::Group> root, const unsigned int numGeometries);
  virtual void initState(DeviceState const& state);

  virtual void updateCamera(const int idCamera, CameraDefinition const& camera);
  virtual void updateLight(const int idLight, LightDefinition const& light);
  virtual void updateMaterial(const int idMaterial, MaterialGUI const& src);
  // B200 extension (the reference rebuilt nothing after initScene): moves instances first .. first + count - 1
  virtual void updateInstanceTransforms(const unsigned int first, const unsigned int count, const float* matrices);
  virtual void rebuildInstanceLevel();
  virtual void updateGeometry(const unsigned int id, const TriangleAttributes* attributes, const size_t numAttributes, const bool rebuild);
  virtual void updateState(DeviceState const& state);

  virtual unsigned int render() = 0;                 // one iteration; returns the iterations done so far
  virtual unsigned int render(const unsigned int count);   // up to `count` iterations in one enqueue

  // Coalescing behind the unchanged `unsigned int render()` (apps/rtigo3/inc/Raytracer.h:79; Application::benchmark calls it
  // once per iteration, Application.cpp:500-503).  The reference's render() only ENQUEUES an asynchronous optixLaunch, so
  // nothing is observable before synchronize() / getOutputBufferHost() / updateDisplayTexture() / an update*().  render()
  // therefore just counts iterations; they are enqueued as ONE batched launch when `limit` of them are pending or at the
  // next of those observation points.  limit 1 = every call launches.  The default comes from initState(): as many
  // iterations as fit the wavefront budget of 64 Mi paths (32 at 1080p), at most 64.
  void setCoalesceLimit(const unsigned int limit) { flush(); m_coalesceLimit = limit ? limit : 1u; m_coalesceExplicit = true; }
  unsigned int getCoalesceLimit() const { return m_coalesceLimit; }
  void flush();                                      // enqueue the pending iterations on all devices
  virtual void updateDisplayTexture() = 0;
  virtual const void* getOutputBufferHost() = 0;

  void getStats(rtc_stats& total);                   // summed over the active devices

  // Sample-range partition across processes.  `id` = the 128 bytes of ncclProcessUniqueId() made on rank 0.
  // Collective; needs exactly one active device.  world == 1 is allowed (the reduce is then the identity).
  void joinProcessGroup(const int rank, const int world, const char id[128]);
  // mean over the ranks of `count` floats at device address src -> dst on rank 0 (0 elsewhere), enqueued on the render
  // stream behind the launches (no host synchronisation).  Collective.  The building block of getOutputBufferHost().
  void reduceMeanToRoot(const uint64_t src, const uint64_t dst, const size_t count);
  // this process's own running average (not a collective); equals getOutputBufferHost() outside a process group
  const void* getLocalOutputBufferHost();
  int getRank() const { return m_rank; }
  int getWorld() const { return m_world; }
  // iterations this process renders: samplesPerPixel / world (joinProcessGroup refuses a count the ranks cannot share equally)
  unsigned int getSamplesPerPixelLocal() const { return samplesPerRank(m_samplesPerPixel, m_world); }
  static unsigned int samplesPerRank(const unsigned int samplesPerPixel, const int world)
  {
    const unsigned int n = samplesPerPixel / (unsigned int)(world > 0 ? world : 1);
    return n ? n : 1u;
  }

public:
  RendererStrategy m_strategy;
  int              m_interop;
  unsigned int     m_tex;
  unsigned int     m_pbo;
  bool m_isValid;
  int                  m_visibleDevices;
  int                  m_deviceOGL;          // always -1 (headless)
  unsigned int         m_activeDevicesMask;
  std::vector<Device*> m_activeDevices;
  unsigned int m_iterationIndex;
  unsigned int m_samplesPerPixel;
  std::vector<unsigned int>       m_peerConnections;
  std::vector< std::vector<int> > m_peerIslands;

protected:
  template <class DeviceType> void createDevices(const int devicesMask, const int miss, const bool onlyFirst);
  unsigned int renderAll(const unsigned int count);
  unsigned int m_pendingFirst = 0, m_pendingCount = 0;   // iterations counted by render() but not yet enqueued
  unsigned int m_coalesceLimit = 1;
  bool         m_coalesceExplicit = false;
  const void* combineProcessGroup();     // the collective behind getOutputBufferHost() when m_world > 1
  void applySeedOffsets();

  int m_rank = 0;
  int m_world = 1;
  struct NcclGroup* m_processGroup = nullptr;
  uint64_t m_combined = 0;               // rank 0: device buffer receiving the mean frame
  size_t   m_combinedPixels = 0;
  void*    m_combinedHost = nullptr;     // rank 0: pinned staging of the mean frame
};

class RaytracerSingleGPU : public Raytracer
{
public:
  RaytracerSingleGPU(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo);
  unsigned int render() override { return renderAll(1); }
  void updateDisplayTexture() override { flush(); m_activeDevices[0]->updateDisplayTexture(); }
  const void* getOutputBufferHost() override { flush(); return (m_processGroup != nullptr) ? combineProcessGroup() : m_activeDevices[0]->getOutputBufferHost(); }
};

class RaytracerMultiGPUZeroCopy : public Raytracer
{
public:
  RaytracerMultiGPUZeroCopy(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo);
  unsigned int render() override { return renderAll(1); }
  void updateDisplayTexture() override { flush(); }
  const void* getOutputBufferHost() override;
};

class RaytracerMultiGPUPeerAccess : public Raytracer
{
public:
  RaytracerMultiGPUPeerAccess(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo);
  ~RaytracerMultiGPUPeerAccess() override;
  unsigned int render() override { return renderAll(1); }
  void updateDisplayTexture() override { flush(); }
  const void* getOutputBufferHost() override;
};

enum CompositeMode { COMPOSITE_PEER_COPY = 0, COMPOSITE_NCCL_REDUCE = 1 };

class RaytracerMultiGPULocalCopy : public Raytracer
{
public:
  RaytracerMultiGPULocalCopy(const int devicesMask, const int miss, const int interop, const unsigned int tex, const unsigned int pbo);
  ~RaytracerMultiGPULocalCopy() override;
  unsigned int render() override { return renderAll(1); }
  void updateDisplayTexture() override { composite(); }
  const void* getOutputBufferHost() override;
  void setCompositeMode(CompositeMode mode) { m_compositeMode = mode; }
private:
  void composite();
  void compositeNccl();
  CompositeMode m_compositeMode = COMPOSITE_PEER_COPY;
  struct NcclState;
  NcclState* m_nccl = nullptr;
};
