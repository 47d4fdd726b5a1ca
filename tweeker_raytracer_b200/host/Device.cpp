// Device.cpp -- base class of the per-GPU devices; see Device.h for the mapping onto the reference.
#include "Device.h"

#include <algorithm>

#include <cmath>
#include <cstring>

#include "Transform.h"

Device::Device(const RendererStrategy strategy, const int ordinal, const int index, const int count, const int miss,
               const int interop, const unsigned int tex, const unsigned int pbo)
: m_strategy(strategy), m_ordinal(ordinal), m_index(index), m_count(count), m_miss(miss), m_interop(interop)
{
  (void)tex; (void)pbo;
  if (interop != 0) std::cerr << "WARNING: Device() OpenGL interop " << interop << " is not available in the headless build, using 0 (host)." << std::endl;
  m_interop = 0;
  RTC_CHECK(rtc_context_create(ordinal, &m_context));

  // Same defaults as Device::Device (apps/rtigo3/src/Device.cpp:280-313).
  std::memset(&m_systemData, 0, sizeof(SystemData));
  m_systemData.resolution = make_int2(1, 1);
  m_systemData.tileSize = make_int2(8, 8);
  m_systemData.tileShift = make_int2(3, 3);
  m_systemData.pathLengths = make_int2(2, 5);
  m_systemData.deviceCount = m_count;
  m_systemData.deviceIndex = m_index;
  m_systemData.distribution = 0;
  m_systemData.samplesSqrt = 1;
  m_systemData.sceneEpsilon = 500.0f * RT_SCENE_EPSILON_SCALE;
  m_systemData.clockScale = 1000.0f * RT_CLOCK_FACTOR_SCALE;
  m_systemData.lensShader = 0;
  m_systemData.envIntegral = 1.0f;
  m_launchWidth = 1;
}

Device::~Device()
{
  if (!m_context) return;
  RTC_CHECK_NO_THROW(rtc_synchronize(m_context));
  auto release = [&](uint64_t& p) { if (p) { RTC_CHECK_NO_THROW(rtc_free(m_context, p)); p = 0; } };
  release(m_systemData.cameraDefinitions);
  release(m_systemData.lightDefinitions);
  release(m_systemData.materialDefinitions);
  release(m_systemData.envTexture);
  release(m_systemData.envCDF_U);
  release(m_systemData.envCDF_V);
  if (m_textureAlbedo) { RTC_CHECK_NO_THROW(rtc_texture_destroy(m_context, m_textureAlbedo)); m_textureAlbedo = 0; }
  if (m_textureCutout) { RTC_CHECK_NO_THROW(rtc_texture_destroy(m_context, m_textureCutout)); m_textureCutout = 0; }
  for (GeometryData& g : m_geometryData) { release(g.d_attributes); release(g.d_indices); }
  if (m_bufferHost) { RTC_CHECK_NO_THROW(rtc_host_free(m_context, m_bufferHost)); m_bufferHost = nullptr; }
  RTC_CHECK_NO_THROW(rtc_context_destroy(m_context));
  m_context = nullptr;
}

static int2 calculateTileShift(const int2 tileSize)
{
  int2 shift = make_int2(0, 0);
  while (shift.x < 32 && (tileSize.x & (1 << shift.x)) == 0) ++shift.x;
  while (shift.y < 32 && (tileSize.y & (1 << shift.y)) == 0) ++shift.y;
  return shift;
}

// Device::initTextures (Device.cpp:910-960): the "albedo" and "cutout" pictures become material textures (the reference
// asserts that both exist; here a missing one just leaves its handle 0), the environment map's texels, CDFs and integral
// go into SystemData.
void Device::initTextures(std::map<std::string, EnvMap*> const& mapOfPictures)
{
  activateContext();
  synchronizeStream();
  auto createTexture = [&](const char* name, uint64_t& handle)
  {
    std::map<std::string, EnvMap*>::const_iterator itp = mapOfPictures.find(std::string(name));
    if (itp == mapOfPictures.end() || itp->second == nullptr || itp->second->getWidth() == 0) return;
    if (handle) { RTC_CHECK(rtc_texture_destroy(m_context, handle)); handle = 0; }
    RTC_CHECK(rtc_texture_create(m_context, itp->second->getWidth(), itp->second->getHeight(), itp->second->getTexels().data(), &handle));
  };
  createTexture("albedo", m_textureAlbedo);
  createTexture("cutout", m_textureCutout);
  std::map<std::string, EnvMap*>::const_iterator it = mapOfPictures.find(std::string("environment"));
  if (it == mapOfPictures.end() || it->second == nullptr) return;
  const EnvMap* env = it->second;
  auto upload = [&](uint64_t& dst, std::vector<float> const& src)
  {
    if (dst) RTC_CHECK(rtc_free(m_context, dst));
    RTC_CHECK(rtc_malloc(m_context, src.size() * sizeof(float), &dst));
    RTC_CHECK(rtc_upload(m_context, dst, src.data(), src.size() * sizeof(float)));
  };
  upload(m_systemData.envTexture, env->getTexels());
  upload(m_systemData.envCDF_U, env->getCDF_U());
  upload(m_systemData.envCDF_V, env->getCDF_V());
  synchronizeStream();
  m_systemData.envWidth = env->getWidth();
  m_systemData.envHeight = env->getHeight();
  m_systemData.envIntegral = env->getIntegral();
  m_isDirtySystemData = true;
}

void Device::initCameras(std::vector<CameraDefinition> const& cameras)
{
  activateContext();
  synchronizeStream();
  const int numCameras = static_cast<int>(cameras.size());
  MY_ASSERT(0 < numCameras);
  if (m_systemData.numCameras != numCameras)
  {
    if (m_systemData.cameraDefinitions) RTC_CHECK(rtc_free(m_context, m_systemData.cameraDefinitions));
    RTC_CHECK(rtc_malloc(m_context, sizeof(CameraDefinition) * numCameras, &m_systemData.cameraDefinitions));
  }
  RTC_CHECK(rtc_upload(m_context, m_systemData.cameraDefinitions, cameras.data(), sizeof(CameraDefinition) * numCameras));
  synchronizeStream();
  m_systemData.numCameras = numCameras;
  m_isDirtySystemData = true;
}

void Device::initLights(std::vector<LightDefinition> const& lights)
{
  activateContext();
  synchronizeStream();
  const int numLights = static_cast<int>(lights.size());
  // numLights is only written when there are lights (Device.cpp:992-996): with none it keeps its default 0.
  if (0 < numLights)
  {
    if (m_systemData.numLights != numLights)
    {
      if (m_systemData.lightDefinitions) RTC_CHECK(rtc_free(m_context, m_systemData.lightDefinitions));
      RTC_CHECK(rtc_malloc(m_context, sizeof(LightDefinition) * numLights, &m_systemData.lightDefinitions));
    }
    RTC_CHECK(rtc_upload(m_context, m_systemData.lightDefinitions, lights.data(), sizeof(LightDefinition) * numLights));
    synchronizeStream();
    m_systemData.numLights = numLights;
  }
  m_isDirtySystemData = true;
}

void Device::convertMaterial(MaterialGUI const& gui, MaterialDefinition& material)
{
  std::memset(&material, 0, sizeof(material));
  material.textureAlbedo = 0;   // device handles are filled in by convertMaterialOnDevice
  material.textureCutout = 0;
  material.roughness = gui.roughness;
  material.indexBSDF = gui.indexBSDF;
  material.albedo = gui.albedo;
  material.absorption = make_float3(0.0f);
  if (0.0f < gui.absorptionScale)
  {
    // effective absorption coefficient: -log(colour) * scale, colour clamped away from zero (Device.cpp:1037-1050)
    const float x = -logf(fmaxf(0.0001f, gui.absorptionColor.x));
    const float y = -logf(fmaxf(0.0001f, gui.absorptionColor.y));
    const float z = -logf(fmaxf(0.0001f, gui.absorptionColor.z));
    material.absorption = make_float3(x, y, z) * gui.absorptionScale;
  }
  material.ior = gui.ior;
  material.flags = gui.thinwalled ? RT_FLAG_THINWALLED : 0u;
}

void Device::convertMaterialOnDevice(MaterialGUI const& gui, MaterialDefinition& material) const
{
  convertMaterial(gui, material);
  material.textureAlbedo = gui.useAlbedoTexture ? m_textureAlbedo : 0;
  material.textureCutout = gui.useCutoutTexture ? m_textureCutout : 0;
}

void Device::updateHitRecords()
{
  if (m_systemData.topObject == 0 || m_instances.empty()) return;
  std::vector<uint32_t> flags(m_instances.size(), 0u);
  bool albedo = false;
  for (MaterialDefinition const& m : m_materials) albedo = albedo || m.textureAlbedo != 0;
  for (size_t i = 0; i < m_instances.size(); ++i)
  {
    const int id = m_instances[i].materialIndex;
    if (0 <= id && (size_t)id < m_materials.size() && m_materials[id].textureCutout != 0) flags[i] = RTC_INSTANCE_CUTOUT;
  }
  RTC_CHECK(rtc_scene_set_instance_flags(m_context, m_systemData.topObject, 0u, (uint32_t)flags.size(), flags.data()));
  RTC_CHECK(rtc_scene_set_albedo_textures(m_context, m_systemData.topObject, albedo ? 1 : 0));
}

void Device::initMaterials(std::vector<MaterialGUI> const& materialsGUI)
{
  activateContext();
  synchronizeStream();
  const int numMaterials = static_cast<int>(materialsGUI.size());
  MY_ASSERT(0 < numMaterials);
  if (m_systemData.numMaterials != numMaterials)
  {
    if (m_systemData.materialDefinitions) RTC_CHECK(rtc_free(m_context, m_systemData.materialDefinitions));
    RTC_CHECK(rtc_malloc(m_context, sizeof(MaterialDefinition) * (numMaterials ? numMaterials : 1), &m_systemData.materialDefinitions));
    m_materials.resize(numMaterials);
  }
  for (int i = 0; i < numMaterials; ++i) convertMaterialOnDevice(materialsGUI[i], m_materials[i]);
  RTC_CHECK(rtc_upload(m_context, m_systemData.materialDefinitions, m_materials.data(), sizeof(MaterialDefinition) * numMaterials));
  synchronizeStream();
  m_systemData.numMaterials = numMaterials;
  m_isDirtySystemData = true;
  updateHitRecords();
}

void Device::initScene(std::shared_ptr<sg::Group> root, const unsigned int numGeometries)
{
  activateContext();
  synchronizeStream();
  // a second initScene replaces the scene: the previous instance level is released (geometries already built are kept and reused)
  if (m_systemData.topObject) { RTC_CHECK(rtc_scene_destroy(m_context, m_systemData.topObject)); m_systemData.topObject = 0; }
  m_geometryData.resize(std::max<size_t>(numGeometries, m_geometryData.size()));
  m_instances.clear();
  float matrix[12] = { 1, 0, 0, 0,  0, 1, 0, 0,  0, 0, 1, 0 };
  InstanceData data;
  traverseNode(root, matrix, data);
  // createTLAS + createHitGroupRecords
  uint64_t top = 0;
  RTC_CHECK(rtc_ias_build(m_context, m_instances.data(), (uint32_t)m_instances.size(), &top));
  m_systemData.topObject = top;
  m_isDirtySystemData = true;
  updateHitRecords();
}

void Device::traverseNode(std::shared_ptr<sg::Node> node, float matrix[12], InstanceData data)
{
  switch (node->getType())
  {
    case sg::NT_GROUP:
    {
      std::shared_ptr<sg::Group> group = std::dynamic_pointer_cast<sg::Group>(node);
      for (size_t i = 0; i < group->getNumChildren(); ++i) traverseNode(group->getChild(i), matrix, data);
      break;
    }
    case sg::NT_INSTANCE:
    {
      std::shared_ptr<sg::Instance> instance = std::dynamic_pointer_cast<sg::Instance>(node);
      float trafo[12];
      multiplyMatrix(trafo, matrix, instance->getTransform());
      if (0 <= instance->getMaterial()) data.idMaterial = instance->getMaterial();
      if (0 <= instance->getLight())    data.idLight = instance->getLight();
      if (instance->getChild()) traverseNode(instance->getChild(), trafo, data);
      break;
    }
    case sg::NT_TRIANGLES:
    {
      std::shared_ptr<sg::Triangles> geometry = std::dynamic_pointer_cast<sg::Triangles>(node);
      data.idGeometry = (int)createGeometry(geometry);
      createInstance(m_geometryData[data.idGeometry].gas, matrix, data);
      break;
    }
  }
}

// One GAS per distinct sg::Triangles (Device.cpp:1333-1425): attributes (48 B stride) and uint3 indices are uploaded
// and stay alive because the per-instance shading table points at them.
unsigned int Device::createGeometry(std::shared_ptr<sg::Triangles> geometry)
{
  const unsigned int id = geometry->getId();
  if (m_geometryData.size() <= id) m_geometryData.resize(id + 1);
  GeometryData& g = m_geometryData[id];
  if (g.built) return id;
  std::vector<TriangleAttributes> const& attributes = geometry->getAttributes();
  std::vector<unsigned int> const& indices = geometry->getIndices();
  g.numAttributes = attributes.size();
  g.numIndices = indices.size();
  RTC_CHECK(rtc_malloc(m_context, sizeof(TriangleAttributes) * attributes.size(), &g.d_attributes));
  RTC_CHECK(rtc_malloc(m_context, sizeof(unsigned int) * indices.size(), &g.d_indices));
  RTC_CHECK(rtc_upload(m_context, g.d_attributes, attributes.data(), sizeof(TriangleAttributes) * attributes.size()));
  RTC_CHECK(rtc_upload(m_context, g.d_indices, indices.data(), sizeof(unsigned int) * indices.size()));
  RTC_CHECK(rtc_synchronize(m_context));
  RTC_CHECK(rtc_gas_build(m_context, g.d_attributes, (uint32_t)sizeof(TriangleAttributes), (uint32_t)attributes.size(),
                          g.d_indices, (uint32_t)(indices.size() / 3), RTC_BUILD_DEFAULT, &g.gas));
  g.built = true;
  return id;
}

void Device::createInstance(const unsigned int gas, float matrix[12], InstanceData const& data)
{
  rtc_instance_desc instance;
  std::memcpy(instance.transform, matrix, sizeof(float) * 12);
  instance.instanceId = (uint32_t)m_instances.size();   // the instance id is its position, as in Device.cpp:1433
  instance.gas = gas;
  instance.materialIndex = data.idMaterial;
  instance.lightIndex = data.idLight;
  m_instances.push_back(instance);
}

void Device::updateCamera(const int idCamera, CameraDefinition const& camera)
{
  activateContext();
  synchronizeStream();
  MY_ASSERT(idCamera < m_systemData.numCameras);
  RTC_CHECK(rtc_upload(m_context, m_systemData.cameraDefinitions + sizeof(CameraDefinition) * idCamera, &camera, sizeof(CameraDefinition)));
  synchronizeStream();
}

void Device::updateLight(const int idLight, LightDefinition const& light)
{
  activateContext();
  synchronizeStream();
  MY_ASSERT(idLight < m_systemData.numLights);
  RTC_CHECK(rtc_upload(m_context, m_systemData.lightDefinitions + sizeof(LightDefinition) * idLight, &light, sizeof(LightDefinition)));
  synchronizeStream();
}

void Device::updateMaterial(const int idMaterial, MaterialGUI const& materialGUI)
{
  activateContext();
  synchronizeStream();
  MY_ASSERT(idMaterial < m_systemData.numMaterials);
  MaterialDefinition& material = m_materials[idMaterial];
  const bool hadCutout = material.textureCutout != 0, hadAlbedo = material.textureAlbedo != 0;
  convertMaterialOnDevice(materialGUI, material);
  RTC_CHECK(rtc_upload(m_context, m_systemData.materialDefinitions + sizeof(MaterialDefinition) * idMaterial, &material, sizeof(MaterialDefinition)));
  synchronizeStream();
  if (hadCutout != (material.textureCutout != 0) || hadAlbedo != (material.textureAlbedo != 0)) updateHitRecords();   // "changeShader", Device.cpp:1111
}

void Device::updateInstanceTransforms(const unsigned int first, const unsigned int count, const float* matrices)
{
  activateContext();
  MY_ASSERT((size_t)first + count <= m_instances.size());
  for (unsigned int i = 0; i < count; ++i) std::memcpy(m_instances[first + i].transform, matrices + 12u * i, sizeof(float) * 12);
  RTC_CHECK(rtc_ias_update(m_context, m_systemData.topObject, first, count, matrices));
}

void Device::rebuildInstanceLevel()
{
  activateContext();
  RTC_CHECK(rtc_ias_rebuild(m_context, m_systemData.topObject));
}

void Device::updateGeometry(const unsigned int id, const TriangleAttributes* attributes, const size_t numAttributes, const bool rebuild)
{
  activateContext();
  MY_ASSERT(id < m_geometryData.size() && m_geometryData[id].built && m_geometryData[id].numAttributes == numAttributes);
  GeometryData& g = m_geometryData[id];
  RTC_CHECK(rtc_upload(m_context, g.d_attributes, attributes, sizeof(TriangleAttributes) * numAttributes));
  if (rebuild) RTC_CHECK(rtc_gas_rebuild(m_context, g.gas, 0));
  else         RTC_CHECK(rtc_gas_refit(m_context, g.gas, 0));
  RTC_CHECK(rtc_ias_update(m_context, m_systemData.topObject, 0, 0, nullptr));
}

void Device::setState(DeviceState const& state)
{
  activateContext();
  synchronizeStream();
  if (m_systemData.resolution != state.resolution)
  {
    m_systemData.resolution = state.resolution;
    m_isDirtyOutputBuffer = true;
    m_isDirtySystemData = true;
  }
  if (m_systemData.tileSize != state.tileSize)
  {
    m_systemData.tileSize = state.tileSize;
    m_systemData.tileShift = calculateTileShift(m_systemData.tileSize);
    m_isDirtySystemData = true;
  }
  m_systemData.distribution = state.distribution;
  m_systemData.samplesSqrt = state.samplesSqrt;
  m_systemData.lensShader = state.lensShader;
  m_systemData.pathLengths = state.pathLengths;
  m_systemData.sceneEpsilon = state.epsilonFactor * RT_SCENE_EPSILON_SCALE;
  m_systemData.envRotation = state.envRotation;
  m_systemData.clockScale = state.clockFactor * RT_CLOCK_FACTOR_SCALE;
  m_isDirtySystemData = true;
}

// Only the local-copy device composites (Device.cpp:1258-1261).
void Device::compositor(Device* other) { (void)other; }

void Device::renderIterations(const unsigned int iterationFirst, const unsigned int count, void** buffer)
{
  for (unsigned int i = 0; i < count; ++i) render(iterationFirst + i, buffer);
}

// The optixLaunch replacement shared by the four strategies.  SystemData travels by value with the launch,
// so the per-iteration "synchronize, then upload iterationIndex" of DeviceSingleGPU.cpp:145-158 has no equivalent.
void Device::launch(const unsigned int launchWidth, const int raygen, const unsigned int iterationFirst, const unsigned int count)
{
  m_systemData.iterationIndex = (int)(m_seedOffset + iterationFirst);
  RTC_CHECK(rtc_launch_ex(m_context, &m_systemData, launchWidth, (uint32_t)m_systemData.resolution.y, raygen, m_miss,
                          (int)(m_seedOffset + iterationFirst), (int)count, (int)iterationFirst, 0));
  m_isDirtySystemData = false;
}

float4* Device::hostBuffer(size_t pixels)
{
  if (m_bufferHostPixels != pixels || m_bufferHost == nullptr)
  {
    if (m_bufferHost) { RTC_CHECK(rtc_synchronize(m_context)); RTC_CHECK(rtc_host_free(m_context, m_bufferHost)); m_bufferHost = nullptr; }
    void* p = nullptr;
    RTC_CHECK(rtc_host_alloc(m_context, sizeof(float4) * (pixels ? pixels : 1), &p));
    m_bufferHost = static_cast<float4*>(p);
    m_bufferHostPixels = pixels;
  }
  return m_bufferHost;
}

void Device::getStats(rtc_stats& stats) const { RTC_CHECK(rtc_stats_get(m_context, &stats)); }
