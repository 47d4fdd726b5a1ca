// Device.h -- one GPU of the renderer, the class the reference calls Device (apps/rtigo3/inc/Device.h:292-420).
// The class shape and virtual interface are kept; everything that was an OptiX or CUDA-driver call in
// apps/rtigo3/src/Device.cpp is a call into the C ABI of librtcore (include/rtc_core.h):
//   ctor            cuCtxCreate/cuStreamCreate/optixDeviceContextCreate/initPipeline (Device.cpp:222-317) -> rtc_context_create
//   initScene       traverseNode/createGeometry/createInstance/createTLAS/createHitGroupRecords (:1058-1532) -> rtc_gas_build, rtc_ias_build
//   render          optixLaunch (DeviceSingleGPU.cpp:164, ...)                                  -> rtc_launch
//   compositor      cuLaunchKernel(compositor) (DeviceMultiGPULocalCopy.cpp:279-337)             -> rtc_composite
// interop / tex / pbo are accepted for signature compatibility and must be 0 (headless).
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "CheckMacros.h"
#include "EnvMap.h"
#include "HostTypes.h"
#include "SceneGraph.h"

struct InstanceData
{
  int idGeometry = -1;
  int idMaterial = -1;
  int idLight = -1;
};

class Device
{
public:
  Device(const RendererStrategy strategy, const int ordinal, const int index, const int count, const int miss,
         const int interop, const unsigned int tex, const unsigned int pbo);
  virtual ~Device();

  virtual void initTextures(std::map<std::string, EnvMap*> const& mapOfPictures);
  virtual void initCameras(std::vector<CameraDefinition> const& cameras);
  virtual void initLights(std::vector<LightDefinition> const& lights);
  virtual void initMaterials(std::vector<MaterialGUI> const& materialsGUI);
  virtual void initScene(std::shared_ptr<sg::Group> root, const unsigned int numGeometries);

  virtual void updateCamera(const int idCamera, CameraDefinition const& camera);
  virtual void updateLight(const int idLight, LightDefinition const& light);
  virtual void updateMaterial(const int idMaterial, MaterialGUI const& materialGUI);
  // B200 extension: object->world matrices (12 floats each) of instances first .. first + count - 1 (the traversal order of
  // initScene); refits the instance level on the device (rtc_ias_update), stream-ordered behind the launches already enqueued
  virtual void updateInstanceTransforms(const unsigned int first, const unsigned int count, const float* matrices);
  virtual void rebuildInstanceLevel();
  // new vertex records (48 B TriangleAttributes, the build's count) of geometry `id` (sg::Triangles id): uploaded into this
  // device's buffer, the GAS refitted (rtc_gas_refit) or rebuilt (rtc_gas_rebuild), the instances updated (rtc_ias_update);
  // all stream-ordered behind the launches already enqueued
  virtual void updateGeometry(const unsigned int id, const TriangleAttributes* attributes, const size_t numAttributes, const bool rebuild);

  virtual void setState(DeviceState const& state);
  virtual void compositor(Device* other);

  virtual void activateContext() = 0;
  virtual void synchronizeStream() = 0;
  virtual void render(const unsigned int iterationIndex, void** buffer) = 0;
  virtual void updateDisplayTexture() = 0;
  virtual const void* getOutputBufferHost() = 0;

  // B200 extension: `count` consecutive iterations in one enqueue (the wavefront keeps several iterations in flight).
  // The default forwards to render() once per iteration.
  virtual void renderIterations(const unsigned int iterationFirst, const unsigned int count, void** buffer);

  // MaterialGUI -> MaterialDefinition (the conversion inside Device::initMaterials, Device.cpp:1024-1052)
  static void convertMaterial(MaterialGUI const& gui, MaterialDefinition& material);

  rtc_context* getContext() const { return m_context; }
  SystemData const& getSystemData() const { return m_systemData; }
  std::vector<MaterialDefinition> const& getMaterials() const { return m_materials; }
  uint64_t getTopObject() const { return m_systemData.topObject; }
  void getStats(rtc_stats& stats) const;
  // B200 extension (sample-range partition, one process per GPU): iteration i of this device draws its seeds from
  // iteration index offset + i, while it is still blended into this device's running average as sample i.
  void setSeedOffset(const unsigned int offset) { m_seedOffset = offset; }
  uint64_t getOutputBufferDevice() const { return m_systemData.outputBuffer; }

protected:
  void traverseNode(std::shared_ptr<sg::Node> node, float matrix[12], InstanceData data);
  unsigned int createGeometry(std::shared_ptr<sg::Triangles> geometry);
  void createInstance(const unsigned int gas, float matrix[12], InstanceData const& data);
  void launch(const unsigned int launchWidth, const int raygen, const unsigned int iterationFirst, const unsigned int count);
  // MaterialGUI -> device MaterialDefinition including the texture handles of this device (Device.cpp:1024-1052, :1112-1113)
  void convertMaterialOnDevice(MaterialGUI const& gui, MaterialDefinition& material) const;
  // createHitGroupRecords (Device.cpp:1492-1532) / the SBT header switch of updateMaterial (:1141-1160): instances whose
  // material has a cutout texture get the cutout hit records
  void updateHitRecords();

public:
  RendererStrategy m_strategy;
  int m_ordinal;
  int m_index;
  int m_count;
  int m_miss;
  int m_interop;

protected:
  struct GeometryData { unsigned int gas = 0; uint64_t d_attributes = 0; uint64_t d_indices = 0; size_t numAttributes = 0; size_t numIndices = 0; bool built = false; };

  rtc_context* m_context = nullptr;
  SystemData   m_systemData;
  bool m_isDirtySystemData = true;
  bool m_isDirtyOutputBuffer = true;
  bool m_ownsSharedBuffer = false;
  int  m_launchWidth = 0;
  unsigned int m_seedOffset = 0;
  uint64_t m_textureAlbedo = 0;   // the reference's m_textureAlbedo / m_textureCutout (Device.h), as rtc_texture handles
  uint64_t m_textureCutout = 0;

  std::vector<GeometryData>      m_geometryData;   // indexed by sg::Triangles id
  std::vector<rtc_instance_desc> m_instances;
  std::vector<MaterialDefinition> m_materials;     // host mirror in device layout
  // host staging of the frame (the reference's std::vector<float4> m_bufferHost, DeviceSingleGPU.h:57), pinned so the
  // device->host copy runs at full PCIe rate and asynchronously
  float4* hostBuffer(size_t pixels);
  float4* m_bufferHost = nullptr;
  size_t  m_bufferHostPixels = 0;
};
