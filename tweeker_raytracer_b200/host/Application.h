// Application.h -- rtigo3's Application (apps/rtigo3/inc/Application.h, src/Application.cpp) re-hosted headless:
// system/scene description loaders (Application.cpp:1046-1299, :1397-1878), createLights (:572-677),
// createCameras (:562-569), the strategy switch (:224-245), render/benchmark (:401-531) and screenshot (:2231-2340).
// GLFW/ImGui/Rasterizer are out of scope; the loaders, index semantics and file formats are kept.
#pragma once
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "Camera.h"
#include "EnvMap.h"
#include "HostTypes.h"
#include "Options.h"
#include "Raytracer.h"
#include "SceneGraph.h"

// Flattened view of the loaded scene (the order Device::traverseNode visits it), used by tools and tests.
struct FlatInstance { float transform[12]; int geometry; int material; int light; };

class Application
{
public:
  // hostOnly = true loads and flattens the scene without creating a Raytracer (no GPU needed; nothing can be rendered).
  explicit Application(Options const& options, bool hostOnly = false);
  ~Application();

  bool isValid() const { return m_isValid; }
  unsigned int render(const unsigned int count = 1);        // advances up to `count` iterations; returns iterations done
  void benchmark();                                         // Application.cpp:491-531: all spp, fps print, tonemapped screenshot
  bool screenshot(const bool tonemap, std::string* writtenPath = nullptr);
  const float* getOutputBufferHost();                       // float4 rows bottom-up, resolution.x * resolution.y
  void tonemapDevice(std::vector<unsigned char>& rgb);      // rtc_tonemap of the current frame (device 0)
  void restartAccumulation();
  // Application::saveSystemDescription (Application.cpp:1302-1345, the 'S' key): writes the current system options in the
  // system description format.  An empty filename yields "system_rtigo3_<date>_<time>.txt" like the reference.
  bool saveSystemDescription(std::string const& filename = std::string(), std::string* writtenPath = nullptr);
  // The GUI mutators of the reference (Application.cpp:410-417, :983, :1003): each restarts the accumulation.
  void setCamera(float phi, float theta, float fov, float distance, const float center[3]);
  bool updateMaterial(int index, MaterialGUI const& material);
  bool updateLightEmission(int index, const float emission[3]);
  // object->world matrix (row-major 3x4) of flattened instance `index` (getFlatInstances); restarts the accumulation
  bool updateInstanceTransform(int index, const float matrix[12]);
  void rebuildInstanceLevel();
  // new vertex records of geometry `index` (the numbering of getGeometries()); false for a bad index or another vertex count
  bool updateGeometry(int index, const TriangleAttributes* attributes, size_t numVerts, bool rebuild);

  // accessors
  Raytracer* getRaytracer() { return m_raytracer.get(); }
  int2 getResolution() const { return m_resolution; }
  // the iterations render() can reach: samplesSqrt^2, or this rank's share of them once the process joined a group
  int getSamplesPerPixel() const { return m_raytracer ? (int)m_raytracer->getSamplesPerPixelLocal() : m_samplesSqrt * m_samplesSqrt; }
  int getMiss() const { return m_miss; }
  int getLightMode() const { return m_light; }
  int getDevicesMask() const { return m_devicesMask; }
  std::string getPrefixScreenshot() const { return m_prefixScreenshot; }
  void getMaterialDefinitions(std::vector<MaterialDefinition>& out) const;
  void getSystemData(int deviceIndex, SystemData& out) const;
  RendererStrategy getStrategy() const { return m_strategy; }
  TonemapperGUI const& getTonemapper() const { return m_tonemapperGUI; }
  DeviceState const& getState() const { return m_state; }
  std::vector<MaterialGUI> const& getMaterialsGUI() const { return m_materialsGUI; }
  std::vector<LightDefinition> const& getLights() const { return m_lights; }
  std::vector<CameraDefinition> const& getCameras() const { return m_cameras; }
  std::vector<std::shared_ptr<sg::Triangles>> const& getGeometries() const { return m_geometries; }
  std::vector<FlatInstance> const& getFlatInstances() const { return m_flatInstances; }
  EnvMap const* getEnvironment() const { return m_environmentMap.get(); }
  EnvMap* getPicture(std::string const& name) const;           // "albedo", "cutout", "environment"; nullptr when absent
  double getLastBenchmarkSeconds() const { return m_benchmarkSeconds; }
  std::string getLastError() const { return m_lastError; }
  void setCompositeMode(int mode);
  // One process per GPU (B200 addition, see Raytracer::joinProcessGroup): this Application becomes rank `rank` of `world`
  // processes rendering disjoint iteration ranges; getOutputBufferHost()/screenshot() are then collectives and rank 0
  // owns the combined frame.  makeProcessGroupId() is called on rank 0; the 128 bytes travel out of band.
  static void makeProcessGroupId(char id[128]);
  bool joinProcessGroup(int rank, int world, const char id[128]);
  // The same, driven by a torchrun-style environment (RANK, WORLD_SIZE, LOCAL_RANK) when RTIGO3_PROCESS_GROUP=1: the id
  // is exchanged through the file RTIGO3_NCCL_ID_FILE (default /tmp/rtigo3_nccl_id_<MASTER_PORT>).  Returns false when
  // the environment does not ask for a process group.
  bool joinProcessGroupFromEnvironment();

private:
  bool loadSystemDescription(std::string const& filename);
  bool loadSceneDescription(std::string const& filename);
  void createCameras();
  void createLights();
  void createPictures();
  void appendInstance(std::shared_ptr<sg::Group>& group, std::shared_ptr<sg::Triangles> geometry, const float trafo[12],
                      std::string const& reference, unsigned int& idInstance);
  std::shared_ptr<sg::Triangles> cachedGeometry(std::string const& key, bool& created);
  // `model assimp <file>` (Assimp.cpp:47-319): Wavefront OBJ through the built-in reader, see MeshImport.cpp
  std::shared_ptr<sg::Group> createASSIMP(std::string const& filename);
  static void calculateTangents(std::vector<TriangleAttributes>& attributes, std::vector<unsigned int> const& indices);
  void flatten(std::shared_ptr<sg::Node> node, const float matrix[12], int material, int light);

private:
  bool m_isValid = false;
  std::string m_lastError;

  // system options (defaults: Application.cpp:55-120)
  RendererStrategy m_strategy = RS_INTERACTIVE_SINGLE_GPU;
  int   m_devicesMask = 255;
  int   m_interop = 0;
  bool  m_present = false;
  int2  m_resolution = { 1, 1 };
  int2  m_tileSize = { 8, 8 };
  int   m_samplesSqrt = 1;
  int   m_miss = 1;
  std::string m_environment;
  float m_environmentRotation = 0.0f;
  float m_clockFactor = 1000.0f;
  int   m_light = 0;
  int2  m_pathLengths = { 0, 2 };
  float m_epsilonFactor = 500.0f;
  LensShader m_lensShader = LENS_SHADER_PINHOLE;
  std::string m_prefixScreenshot = "./img";
  // the reference hard-codes these two file names (Application.cpp:684, :688); extension keywords "textureAlbedo" /
  // "textureCutout" override them.  Unreadable or missing files fall back to procedural pictures.
  std::string m_fileAlbedo = "./NVIDIA_Logo.jpg";
  std::string m_fileCutout = "./slots_alpha.png";
  TonemapperGUI m_tonemapperGUI;
  int   m_compositeMode = 0;     // extension keyword "composite": 0 peer copies, 1 NCCL reduce (local-copy strategy)
  int   m_batch = 1;             // extension keyword "batchIterations": iterations per enqueue in benchmark()
  int   m_coalesce = 0;          // extension keyword "coalesceIterations": Raytracer::setCoalesceLimit (0 = its default, 1 = every render() launches)

  Camera m_camera;
  DeviceState m_state;
  std::unique_ptr<Raytracer> m_raytracer;

  std::shared_ptr<sg::Group> m_scene;
  unsigned int m_idGroup = 0, m_idInstance = 0, m_idGeometry = 0;
  std::vector<std::shared_ptr<sg::Triangles>> m_geometries;
  std::map<std::string, unsigned int> m_mapGeometries;
  std::map<std::string, std::shared_ptr<sg::Group>> m_mapGroups;    // imported models by file name
  std::vector<MaterialGUI> m_materialsGUI;
  std::map<std::string, int> m_mapMaterialReferences;
  std::vector<CameraDefinition> m_cameras;
  std::vector<LightDefinition> m_lights;
  std::unique_ptr<EnvMap> m_environmentMap, m_pictureAlbedo, m_pictureCutout;
  std::map<std::string, EnvMap*> m_mapPictures;
  std::vector<FlatInstance> m_flatInstances;
  double m_benchmarkSeconds = 0.0;
};
