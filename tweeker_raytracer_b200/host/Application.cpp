// Application.cpp -- headless re-hosting of rtigo3's Application; see Application.h.
#include "Application.h"

#include <fcntl.h>
#include <sys/stat.h>
#include <sys/types.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <functional>
#include <iomanip>
#include <iostream>
#include <sstream>
#include <stack>

#include "ImageIO.h"
#include "NcclComposite.h"
#include "Parser.h"
#include "Transform.h"

static int envInt(const char* name, int fallback)
{
  const char* v = std::getenv(name);
  return (v && *v) ? std::atoi(v) : fallback;
}

static const float kIdentity12[12] = { 1, 0, 0, 0,  0, 1, 0, 0,  0, 0, 1, 0 };

Application::Application(Options const& options, bool hostOnly)
{
  // neutral tonemapper (Application.cpp:100-110)
  m_tonemapperGUI.gamma = 2.2f;
  m_tonemapperGUI.colorBalance[0] = m_tonemapperGUI.colorBalance[1] = m_tonemapperGUI.colorBalance[2] = 1.0f;
  m_tonemapperGUI.whitePoint = 1.0f;
  m_tonemapperGUI.burnHighlights = 0.8f;
  m_tonemapperGUI.crushBlacks = 0.2f;
  m_tonemapperGUI.saturation = 1.2f;
  m_tonemapperGUI.brightness = 0.8f;

  try
  {
    if (!loadSystemDescription(options.getSystem()))
    {
      m_lastError = "failed to load system description file " + options.getSystem();
      std::cerr << "ERROR: Application() " << m_lastError << std::endl;
      return;
    }
    m_camera.setResolution(m_resolution.x, m_resolution.y);

    // one process per GPU: this process drives the GPU of its LOCAL_RANK as a single-GPU renderer (joined below)
    const bool processGroup = !hostOnly && envInt("RTIGO3_PROCESS_GROUP", 0) == 1 && 1 < envInt("WORLD_SIZE", 1);
    if (processGroup)
    {
      m_strategy = RS_INTERACTIVE_SINGLE_GPU;
      m_devicesMask = 1 << envInt("LOCAL_RANK", envInt("RANK", 0));
    }

    // strategy switch (Application.cpp:224-245); distribution = 1 for the multi-GPU strategies
    switch (hostOnly ? NUM_RENDERER_STRATEGIES : m_strategy)
    {
      case RS_INTERACTIVE_SINGLE_GPU:
        m_raytracer = std::make_unique<RaytracerSingleGPU>(m_devicesMask, m_miss, m_interop, 0u, 0u);
        m_state.distribution = 0;
        break;
      case RS_INTERACTIVE_MULTI_GPU_ZERO_COPY:
        m_raytracer = std::make_unique<RaytracerMultiGPUZeroCopy>(m_devicesMask, m_miss, m_interop, 0u, 0u);
        m_state.distribution = 1;
        break;
      case RS_INTERACTIVE_MULTI_GPU_PEER_ACCESS:
        m_raytracer = std::make_unique<RaytracerMultiGPUPeerAccess>(m_devicesMask, m_miss, m_interop, 0u, 0u);
        m_state.distribution = 1;
        break;
      case RS_INTERACTIVE_MULTI_GPU_LOCAL_COPY:
      {
        RaytracerMultiGPULocalCopy* rt = new RaytracerMultiGPULocalCopy(m_devicesMask, m_miss, m_interop, 0u, 0u);
        rt->setCompositeMode(m_compositeMode ? COMPOSITE_NCCL_REDUCE : COMPOSITE_PEER_COPY);
        m_raytracer.reset(rt);
        m_state.distribution = 1;
        break;
      }
      default:
        break;
    }
    if (hostOnly)
    {
      m_state.distribution = (m_strategy == RS_INTERACTIVE_SINGLE_GPU) ? 0 : 1;
    }
    else if (!m_raytracer || !m_raytracer->m_isValid)
    {
      m_lastError = "could not initialize Raytracer (no active device in devicesMask?)";
      std::cerr << "ERROR: Application() " << m_lastError << std::endl;
      return;
    }

    m_state.resolution    = m_resolution;
    m_state.tileSize      = m_tileSize;
    m_state.pathLengths   = m_pathLengths;
    m_state.samplesSqrt   = m_samplesSqrt;
    m_state.lensShader    = m_lensShader;
    m_state.epsilonFactor = m_epsilonFactor;
    m_state.envRotation   = m_environmentRotation;
    m_state.clockFactor   = m_clockFactor;
    if (m_raytracer)
    {
      if (0 < m_coalesce) m_raytracer->setCoalesceLimit((unsigned int)m_coalesce);
      m_raytracer->initState(m_state);
    }

    m_scene = std::make_shared<sg::Group>(m_idGroup++);
    createCameras();
    createLights();     // NOTE: before the scene file is read -> the area light owns material 0 / geometry 0 / instance 0
    createPictures();

    if (!loadSceneDescription(options.getScene()))
    {
      m_lastError = "failed to load scene description file " + options.getScene();
      std::cerr << "ERROR: Application() " << m_lastError << std::endl;
      return;
    }
    if (m_materialsGUI.empty())   // the reference asserts on this (Device.cpp:1008)
    {
      MaterialGUI fallback; fallback.name = "default";
      m_mapMaterialReferences["default"] = 0;
      m_materialsGUI.push_back(fallback);
    }
    m_flatInstances.clear();
    flatten(m_scene, kIdentity12, -1, -1);

    if (hostOnly) { m_isValid = true; return; }

    m_raytracer->initTextures(m_mapPictures);
    m_raytracer->initCameras(m_cameras);
    m_raytracer->initLights(m_lights);
    m_raytracer->initMaterials(m_materialsGUI);
    m_raytracer->initScene(m_scene, m_idGeometry);
    m_isValid = true;
    if (processGroup && !joinProcessGroupFromEnvironment()) m_isValid = false;
  }
  catch (std::exception const& e)
  {
    m_lastError = e.what();
    std::cerr << e.what() << std::endl;
  }
}

Application::~Application() {}

void Application::makeProcessGroupId(char id[128]) { ncclProcessUniqueId(id); }

bool Application::joinProcessGroup(int rank, int world, const char id[128])
{
  try { m_raytracer->joinProcessGroup(rank, world, id); return true; }
  catch (std::exception const& e) { m_lastError = e.what(); std::cerr << e.what() << std::endl; return false; }
}

// Rendezvous of `rtigo3_b200` launched torchrun-style (RTIGO3_PROCESS_GROUP=1): rank 0 hands the 128-byte NCCL id to the
// other ranks through a file.  The file is private to the job: its name carries a nonce (TORCHELASTIC_RUN_ID when the
// launcher sets one, else MASTER_PORT + the launcher's pid, which all ranks share), it is created with O_EXCL | O_NOFOLLOW
// and mode 0600 after any stale file of that name was unlinked, and it starts with a magic word + the nonce, which the
// readers verify together with the owner (a stale or foreign file is never taken for this job's id).
bool Application::joinProcessGroupFromEnvironment()
{
  const int world = envInt("WORLD_SIZE", 1), rank = envInt("RANK", 0);
  if (envInt("RTIGO3_PROCESS_GROUP", 0) != 1 || world < 2) return false;
  std::string nonce;
  if (const char* run = std::getenv("TORCHELASTIC_RUN_ID")) nonce = run;
  nonce += "_" + std::to_string(envInt("MASTER_PORT", 0)) + "_" + std::to_string((long)getppid());
  for (char& c : nonce) if (!(std::isalnum((unsigned char)c) || c == '_' || c == '-')) c = '_';
  const char* dir = std::getenv("XDG_RUNTIME_DIR");
  std::string file = std::string(dir && *dir ? dir : "/tmp") + "/rtigo3_nccl_id_" + std::to_string((long)geteuid()) + "_" + nonce;
  if (const char* f = std::getenv("RTIGO3_NCCL_ID_FILE")) file = f;
  struct Header { char magic[8]; char nonce[56]; } want;
  std::memset(&want, 0, sizeof(want));
  std::memcpy(want.magic, "RTIGO3ID", 8);
  std::strncpy(want.nonce, nonce.c_str(), sizeof(want.nonce) - 1);
  char id[128];
  if (rank == 0)
  {
    makeProcessGroupId(id);
    const std::string tmp = file + ".tmp";
    ::unlink(file.c_str());
    ::unlink(tmp.c_str());
    const int fd = ::open(tmp.c_str(), O_CREAT | O_EXCL | O_WRONLY | O_NOFOLLOW, 0600);
    bool ok = fd >= 0 && ::write(fd, &want, sizeof(want)) == (ssize_t)sizeof(want) && ::write(fd, id, sizeof(id)) == (ssize_t)sizeof(id);
    if (fd >= 0) ok = (::close(fd) == 0) && ok;
    if (!ok) { m_lastError = "cannot write " + tmp; std::cerr << "ERROR: " << m_lastError << std::endl; return false; }
    if (std::rename(tmp.c_str(), file.c_str()) != 0) { m_lastError = "cannot rename " + tmp; return false; }
  }
  else
  {
    // the rename makes the file appear complete; wait for it for up to two minutes
    bool got = false;
    for (int attempt = 0; attempt < 2400 && !got; ++attempt)
    {
      const int fd = ::open(file.c_str(), O_RDONLY | O_NOFOLLOW);
      if (fd >= 0)
      {
        struct stat st;
        Header have;
        got = ::fstat(fd, &st) == 0 && st.st_uid == geteuid() && S_ISREG(st.st_mode)
           && ::read(fd, &have, sizeof(have)) == (ssize_t)sizeof(have) && std::memcmp(&have, &want, sizeof(want)) == 0
           && ::read(fd, id, sizeof(id)) == (ssize_t)sizeof(id);
        ::close(fd);
      }
      if (!got) { struct timespec ts = { 0, 50 * 1000 * 1000 }; nanosleep(&ts, nullptr); }
    }
    if (!got) { m_lastError = "timed out waiting for " + file; std::cerr << "ERROR: " << m_lastError << std::endl; return false; }
  }
  const bool ok = joinProcessGroup(rank, world, id);
  if (rank == 0) ::unlink(file.c_str());   // every rank has read it once ncclCommInitRank returned (or the join failed: do not leave it behind)
  return ok;
}

void Application::setCompositeMode(int mode)
{
  m_compositeMode = mode;
  if (m_strategy == RS_INTERACTIVE_MULTI_GPU_LOCAL_COPY && m_raytracer)
    static_cast<RaytracerMultiGPULocalCopy*>(m_raytracer.get())->setCompositeMode(mode ? COMPOSITE_NCCL_REDUCE : COMPOSITE_PEER_COPY);
}

void Application::getMaterialDefinitions(std::vector<MaterialDefinition>& out) const
{
  out.resize(m_materialsGUI.size());
  for (size_t i = 0; i < m_materialsGUI.size(); ++i)
  {
    Device::convertMaterial(m_materialsGUI[i], out[i]);
    // HOST handles (address of header + texels), valid while this Application lives: what a CPU checker dereferences
    if (m_materialsGUI[i].useAlbedoTexture && m_pictureAlbedo) out[i].textureAlbedo = (uint64_t)(uintptr_t)m_pictureAlbedo->getHandleBlob().data();
    if (m_materialsGUI[i].useCutoutTexture && m_pictureCutout) out[i].textureCutout = (uint64_t)(uintptr_t)m_pictureCutout->getHandleBlob().data();
  }
}

// SystemData of one active device; in host-only mode the value fields are derived the way Device::setState does
// (pointers stay null, deviceCount = 1).
void Application::getSystemData(int deviceIndex, SystemData& out) const
{
  if (m_raytracer && deviceIndex >= 0 && (size_t)deviceIndex < m_raytracer->m_activeDevices.size())
  {
    out = m_raytracer->m_activeDevices[deviceIndex]->getSystemData();
    return;
  }
  std::memset(&out, 0, sizeof(out));
  out.resolution = m_state.resolution; out.tileSize = m_state.tileSize;
  int sx = 0, sy = 0;
  while (sx < 32 && (m_state.tileSize.x & (1 << sx)) == 0) ++sx;
  while (sy < 32 && (m_state.tileSize.y & (1 << sy)) == 0) ++sy;
  out.tileShift = make_int2(sx, sy);
  out.pathLengths = m_state.pathLengths; out.deviceCount = 1; out.deviceIndex = 0; out.distribution = m_state.distribution;
  out.samplesSqrt = m_state.samplesSqrt; out.sceneEpsilon = m_state.epsilonFactor * RT_SCENE_EPSILON_SCALE;
  out.clockScale = m_state.clockFactor * RT_CLOCK_FACTOR_SCALE; out.lensShader = m_state.lensShader;
  out.numCameras = (int)m_cameras.size(); out.numMaterials = (int)m_materialsGUI.size(); out.numLights = (int)m_lights.size();
  out.envRotation = m_state.envRotation; out.envIntegral = 1.0f;
  if (m_environmentMap && m_mapPictures.count("environment"))
  { out.envWidth = m_environmentMap->getWidth(); out.envHeight = m_environmentMap->getHeight(); out.envIntegral = m_environmentMap->getIntegral(); }
}

bool Application::saveSystemDescription(std::string const& filename, std::string* writtenPath)
{
  std::ostringstream d;
  d << "strategy " << (int)m_strategy << '\n' << "devicesMask " << m_devicesMask << '\n' << "interop " << m_interop << '\n'
    << "present " << (m_present ? "1" : "0") << '\n' << "resolution " << m_resolution.x << " " << m_resolution.y << '\n'
    << "tileSize " << m_tileSize.x << " " << m_tileSize.y << '\n' << "samplesSqrt " << m_samplesSqrt << '\n' << "miss " << m_miss << '\n';
  if (!m_environment.empty()) d << "envMap " << m_environment << '\n';
  d << "envRotation " << m_environmentRotation << '\n' << "clockFactor " << m_clockFactor << '\n' << "light " << m_light << '\n'
    << "pathLengths " << m_pathLengths.x << " " << m_pathLengths.y << '\n' << "epsilonFactor " << m_epsilonFactor << '\n'
    << "lensShader " << (int)m_lensShader << '\n'
    << "center " << m_camera.m_center.x << " " << m_camera.m_center.y << " " << m_camera.m_center.z << '\n'
    << "camera " << m_camera.m_phi << " " << m_camera.m_theta << " " << m_camera.m_fov << " " << m_camera.m_distance << '\n';
  if (!m_prefixScreenshot.empty()) d << "prefixScreenshot " << m_prefixScreenshot << '\n';
  d << "gamma " << m_tonemapperGUI.gamma << '\n'
    << "colorBalance " << m_tonemapperGUI.colorBalance[0] << " " << m_tonemapperGUI.colorBalance[1] << " " << m_tonemapperGUI.colorBalance[2] << '\n'
    << "whitePoint " << m_tonemapperGUI.whitePoint << '\n' << "burnHighlights " << m_tonemapperGUI.burnHighlights << '\n'
    << "crushBlacks " << m_tonemapperGUI.crushBlacks << '\n' << "saturation " << m_tonemapperGUI.saturation << '\n'
    << "brightness " << m_tonemapperGUI.brightness << '\n';
  if (m_compositeMode) d << "composite " << m_compositeMode << '\n';
  if (m_batch != 1) d << "batchIterations " << m_batch << '\n';
  if (m_coalesce != 0) d << "coalesceIterations " << m_coalesce << '\n';
  if (m_fileAlbedo != "./NVIDIA_Logo.jpg") d << "textureAlbedo " << m_fileAlbedo << '\n';
  if (m_fileCutout != "./slots_alpha.png") d << "textureCutout " << m_fileCutout << '\n';
  std::string path = filename;
  if (path.empty())
  {
    const std::time_t now = std::time(nullptr);
    std::tm tmv; localtime_r(&now, &tmv);
    std::ostringstream name; name << "system_rtigo3_" << std::put_time(&tmv, "%Y%m%d_%H%M%S") << ".txt";
    path = name.str();
  }
  FILE* f = std::fopen(path.c_str(), "w");
  if (!f) return false;
  const std::string text = d.str();
  const bool ok = std::fwrite(text.data(), 1, text.size(), f) == text.size();
  std::fclose(f);
  if (ok) std::cout << path << std::endl;
  if (writtenPath) *writtenPath = ok ? path : std::string();
  return ok;
}

void Application::setCamera(float phi, float theta, float fov, float distance, const float center[3])
{
  m_camera.m_phi = phi; m_camera.m_theta = theta; m_camera.m_fov = fov; m_camera.m_distance = distance;
  m_camera.m_center = make_float3(center[0], center[1], center[2]);
  m_camera.markDirty();
  CameraDefinition camera;
  if (m_camera.getFrustum(camera.P, camera.U, camera.V, camera.W))
  {
    m_cameras[0] = camera;
    if (m_raytracer) m_raytracer->updateCamera(0, camera);
  }
}

bool Application::updateMaterial(int index, MaterialGUI const& material)
{
  if (index < 0 || (size_t)index >= m_materialsGUI.size()) return false;
  const std::string name = m_materialsGUI[index].name;
  m_materialsGUI[index] = material;
  m_materialsGUI[index].name = name;
  if (m_raytracer) m_raytracer->updateMaterial(index, m_materialsGUI[index]);
  return true;
}

bool Application::updateLightEmission(int index, const float emission[3])
{
  if (index < 0 || (size_t)index >= m_lights.size()) return false;
  m_lights[index].emission = make_float3(emission[0], emission[1], emission[2]);
  if (m_raytracer) m_raytracer->updateLight(index, m_lights[index]);
  return true;
}

bool Application::updateInstanceTransform(int index, const float matrix[12])
{
  if (index < 0 || (size_t)index >= m_flatInstances.size()) return false;
  std::memcpy(m_flatInstances[index].transform, matrix, sizeof(float) * 12);
  if (m_raytracer) m_raytracer->updateInstanceTransforms((unsigned int)index, 1u, matrix);
  return true;
}

void Application::rebuildInstanceLevel() { if (m_raytracer) m_raytracer->rebuildInstanceLevel(); }

bool Application::updateGeometry(int index, const TriangleAttributes* attributes, size_t numVerts, bool rebuild)
{
  if (index < 0 || (size_t)index >= m_geometries.size()) return false;
  sg::Triangles& t = *m_geometries[index];
  if (numVerts != t.getAttributes().size()) return false;
  t.setAttributes(std::vector<TriangleAttributes>(attributes, attributes + numVerts));
  if (m_raytracer) m_raytracer->updateGeometry(t.getId(), t.getAttributes().data(), numVerts, rebuild);
  return true;
}

void Application::restartAccumulation() { if (m_raytracer) m_raytracer->updateState(m_state); }

unsigned int Application::render(const unsigned int count)
{
  try { return m_raytracer->render(count); }
  catch (std::exception const& e) { m_lastError = e.what(); std::cerr << e.what() << std::endl; m_isValid = false; return 0; }
}

// Application::benchmark (Application.cpp:491-531)
void Application::benchmark()
{
  try
  {
    const unsigned int spp = m_raytracer->getSamplesPerPixelLocal();   // samplesSqrt^2, or this rank's share of it
    const auto t0 = std::chrono::steady_clock::now();
    unsigned int iterationIndex = 0;
    while (iterationIndex < spp) iterationIndex = m_raytracer->render((unsigned int)std::max(1, m_batch));
    m_raytracer->synchronize();
    m_benchmarkSeconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    const double fps = double(iterationIndex) / m_benchmarkSeconds;
    std::ostringstream stream;
    stream.precision(3);
    stream << std::fixed << iterationIndex << " / " << m_benchmarkSeconds << " = " << fps << " fps";
    if (1 < m_raytracer->getWorld())   // one process per GPU: this rank's share of the samples
      stream << " (rank " << m_raytracer->getRank() << " of " << m_raytracer->getWorld() << ": " << iterationIndex * (unsigned int)m_raytracer->getWorld() << " spp in the combined frame)";
    std::cout << stream.str() << std::endl;
    screenshot(true);
  }
  catch (std::exception const& e) { m_lastError = e.what(); std::cerr << e.what() << std::endl; }
}

const float* Application::getOutputBufferHost()
{
  try { return reinterpret_cast<const float*>(m_raytracer->getOutputBufferHost()); }
  catch (std::exception const& e) { m_lastError = e.what(); std::cerr << e.what() << std::endl; return nullptr; }
}

// The tonemapper of Application::screenshot (Application.cpp:2262-2295) as a device kernel, which the reference
// leaves as a to-do ("PERF Add a native CUDA kernel doing this", :2275).
void Application::tonemapDevice(std::vector<unsigned char>& rgb)
{
  const size_t pixels = (size_t)m_resolution.x * (size_t)m_resolution.y;
  rgb.resize(3 * pixels);
  const float* host = getOutputBufferHost();      // collective in a process group; only rank 0 holds the frame
  if (!host) return;
  Device* device = m_raytracer->m_activeDevices[0];
  rtc_context* ctx = device->getContext();
  uint64_t d_rgba = 0, d_rgb = 0;
  RTC_CHECK(rtc_malloc(ctx, pixels * 16, &d_rgba));
  RTC_CHECK(rtc_malloc(ctx, pixels * 3, &d_rgb));
  RTC_CHECK(rtc_upload(ctx, d_rgba, host, pixels * 16));
  RTC_CHECK(rtc_tonemap(ctx, &m_tonemapperGUI, d_rgba, d_rgb, pixels));
  RTC_CHECK(rtc_download(ctx, rgb.data(), d_rgb, pixels * 3));
  RTC_CHECK(rtc_synchronize(ctx));
  RTC_CHECK(rtc_free(ctx, d_rgba));
  RTC_CHECK(rtc_free(ctx, d_rgb));
}

bool Application::screenshot(const bool tonemap, std::string* writtenPath)
{
  try
  {
    std::ostringstream path;
    const std::time_t now = std::time(nullptr);
    std::tm tmv; localtime_r(&now, &tmv);
    // in a process group the combined frame holds every rank's samples: world x the local count
    path << m_prefixScreenshot << "_" << m_raytracer->m_iterationIndex * (unsigned int)std::max(1, m_raytracer->getWorld()) << "spp_" << std::put_time(&tmv, "%Y%m%d_%H%M%S");
    bool ok = false;
    std::string file;
    const bool writer = m_raytracer->getRank() == 0;    // in a process group fetching the frame is a collective; rank 0 owns the result
    if (tonemap)
    {
      std::vector<unsigned char> rgb;
      tonemapDevice(rgb);
      file = path.str() + ".png";
      ok = !writer || writePNG(file, m_resolution.x, m_resolution.y, rgb.data(), true);   // frame rows are bottom-up
    }
    else
    {
      const float* host = getOutputBufferHost();      // nullptr on the other ranks of a process group
      file = path.str() + ".hdr";
      ok = !writer || (host && writeHDR(file, m_resolution.x, m_resolution.y, host, true));
    }
    if (!writer) { if (writtenPath) writtenPath->clear(); return ok; }
    if (ok) std::cout << file << std::endl;
    if (writtenPath) *writtenPath = ok ? file : std::string();
    return ok;
  }
  catch (std::exception const& e) { m_lastError = e.what(); std::cerr << e.what() << std::endl; return false; }
}

void Application::createCameras()
{
  CameraDefinition camera;
  m_camera.getFrustum(camera.P, camera.U, camera.V, camera.W, true);
  m_cameras.push_back(camera);
}

// Application::createLights (Application.cpp:572-677): the environment light (miss 1|2) is light 0, the optional
// area light follows; its quad, material "rtigo3_area_light" and instance are created here, ahead of the scene file.
void Application::createLights()
{
  LightDefinition light;
  std::memset(&light, 0, sizeof(light));
  light.position = make_float3(0.0f, 0.0f, 0.0f);
  light.vecU     = make_float3(1.0f, 0.0f, 0.0f);
  light.vecV     = make_float3(0.0f, 1.0f, 0.0f);
  light.normal   = make_float3(0.0f, 0.0f, 1.0f);
  light.area     = 1.0f;
  light.emission = make_float3(1.0f, 1.0f, 1.0f);

  if (m_miss == 1 || m_miss == 2)
  {
    light.type = RT_LIGHT_ENVIRONMENT;
    light.area = 4.0f * RT_PI_F;
    m_lights.push_back(light);
  }

  const int indexLight = static_cast<int>(m_lights.size());
  if (m_light == 1 || m_light == 2)
  {
    const float half = (m_light == 1) ? 0.5f : 2.0f;      // 1x1 quad at y = 1.95, or 4x4 quad at y = 4
    const float y    = (m_light == 1) ? 1.95f : 4.0f;
    light.type     = RT_LIGHT_PARALLELOGRAM;
    light.position = make_float3(-half, y, -half);
    light.vecU     = make_float3(2.0f * half, 0.0f, 0.0f);
    light.vecV     = make_float3(0.0f, 0.0f, 2.0f * half);
    const float3 n = cross(light.vecU, light.vecV);
    light.area     = length(n);
    light.normal   = n / light.area;
    light.emission = make_float3(10.0f);
    m_lights.push_back(light);

    const std::string reference("rtigo3_area_light");
    const int indexMaterial = static_cast<int>(m_materialsGUI.size());
    MaterialGUI materialGUI;
    materialGUI.name = reference;
    materialGUI.indexBSDF = INDEX_BRDF_SPECULAR;
    materialGUI.albedo = make_float3(0.0f);
    materialGUI.roughness = make_float2(0.1f, 0.1f);
    materialGUI.absorptionColor = make_float3(1.0f);
    materialGUI.absorptionScale = 0.0f;
    materialGUI.ior = 1.5f;
    materialGUI.thinwalled = true;
    m_materialsGUI.push_back(materialGUI);
    m_mapMaterialReferences[reference] = indexMaterial;

    m_mapGeometries[reference] = m_idGeometry;
    std::shared_ptr<sg::Triangles> geometry(new sg::Triangles(m_idGeometry++));
    geometry->createParallelogram(light.position, light.vecU, light.vecV, light.normal);
    m_geometries.push_back(geometry);

    std::shared_ptr<sg::Instance> instance(new sg::Instance(m_idInstance++));
    instance->setChild(geometry);
    instance->setMaterial(indexMaterial);
    instance->setLight(indexLight);
    m_scene->addChild(instance);
  }
}

// Only the environment map is created: the reference's two hard-coded material images are not sampled unless the GUI
// enables them (Application.cpp:679-699, :1560-1561) and are treated as absent.  `envMap procedural [w h]` (or a
// missing file) yields the analytic map of EnvMap::createProcedural.
EnvMap* Application::getPicture(std::string const& name) const
{
  std::map<std::string, EnvMap*>::const_iterator it = m_mapPictures.find(name);
  return (it == m_mapPictures.end()) ? nullptr : it->second;
}

// Application::createPictures (Application.cpp:679-699): the "albedo" and "cutout" pictures always exist (the materials
// refer to them once the GUI toggles are set), the environment only for miss 2.
void Application::createPictures()
{
  auto picture = [&](std::unique_ptr<EnvMap>& slot, std::string const& file, const char* name, bool cutout)
  {
    slot.reset(new EnvMap());
    if (!slot->loadImage(file))
    {
      if (FILE* f = std::fopen(file.c_str(), "rb"))
      {
        std::fclose(f);
        std::cerr << "WARNING: createPictures() could not decode " << file << " (PNG, PGM/PPM and .hdr are supported), using the procedural " << name << " picture." << std::endl;
      }
      if (cutout) slot->createCutoutProcedural(256, 256); else slot->createAlbedoProcedural(256, 256);
    }
    m_mapPictures[std::string(name)] = slot.get();
  };
  picture(m_pictureAlbedo, m_fileAlbedo, "albedo", false);
  picture(m_pictureCutout, m_fileCutout, "cutout", true);
  if (m_miss != 2) return;
  m_environmentMap.reset(new EnvMap());
  bool ok = false;
  unsigned int w = 2048, h = 1024;
  if (!m_environment.empty() && m_environment.compare(0, 10, "procedural") != 0)
  {
    ok = m_environmentMap->loadHDR(m_environment);
    if (!ok) std::cerr << "WARNING: createPictures() could not read " << m_environment << ", using the procedural environment." << std::endl;
  }
  else if (m_environment.size() > 10)
  {
    unsigned int pw = 0, ph = 0;
    if (std::sscanf(m_environment.c_str() + 10, "%u %u", &pw, &ph) == 2 && pw >= 2 && ph >= 2) { w = pw; h = ph; }
  }
  if (!ok) ok = m_environmentMap->createProcedural(w, h);
  if (ok) m_mapPictures[std::string("environment")] = m_environmentMap.get();
}

// ------------------------------------------------------------------------------------------------------------------
// System description (Application.cpp:1046-1299): keyword followed by its values; unknown keywords only warn.
// ------------------------------------------------------------------------------------------------------------------
bool Application::loadSystemDescription(std::string const& filename)
{
  Parser parser;
  if (!parser.load(filename)) return false;

  std::string token;
  ParserTokenType tokenType;
  auto nextInt = [&]() { parser.getNextToken(token); return std::atoi(token.c_str()); };
  auto nextFloat = [&]() { parser.getNextToken(token); return (float)std::atof(token.c_str()); };

  std::map<std::string, std::function<void()>> keywords;
  keywords["strategy"] = [&]() {
    const int strategy = nextInt();
    if (0 <= strategy && strategy < NUM_RENDERER_STRATEGIES) m_strategy = static_cast<RendererStrategy>(strategy);
    else std::cerr << "WARNING: loadSystemDescription() Invalid renderer strategy " << strategy << ", using Interactive Single GPU." << std::endl;
  };
  keywords["devicesMask"] = [&]() { m_devicesMask = nextInt(); };
  keywords["interop"] = [&]() {
    m_interop = nextInt();
    if (m_interop < 0 || 2 < m_interop) { std::cerr << "WARNING: loadSystemDescription() Invalid interop value " << m_interop << ", using interop 0 (host)." << std::endl; m_interop = 0; }
  };
  keywords["present"] = [&]() { m_present = (nextInt() != 0); };
  keywords["resolution"] = [&]() { m_resolution.x = std::max(1, nextInt()); m_resolution.y = std::max(1, nextInt()); };
  keywords["tileSize"] = [&]() {
    m_tileSize.x = std::max(1, nextInt()); m_tileSize.y = std::max(1, nextInt());
    if (m_tileSize.x & (m_tileSize.x - 1)) { std::cerr << "ERROR: loadSystemDescription(): tileSize.x = " << m_tileSize.x << " is not power-of-two, using 8." << std::endl; m_tileSize.x = 8; }
    if (m_tileSize.y & (m_tileSize.y - 1)) { std::cerr << "ERROR: loadSystemDescription(): tileSize.y = " << m_tileSize.y << " is not power-of-two, using 8." << std::endl; m_tileSize.y = 8; }
  };
  keywords["samplesSqrt"] = [&]() { m_samplesSqrt = std::max(1, nextInt()); };
  keywords["miss"] = [&]() { m_miss = nextInt(); };
  keywords["envMap"] = [&]() { parser.getNextLine(token); m_environment = token; };
  keywords["envRotation"] = [&]() { m_environmentRotation = nextFloat(); };
  keywords["clockFactor"] = [&]() { m_clockFactor = nextFloat(); };
  keywords["light"] = [&]() { m_light = std::min(2, std::max(0, nextInt())); };
  keywords["pathLengths"] = [&]() { m_pathLengths.x = nextInt(); m_pathLengths.y = nextInt(); };
  keywords["epsilonFactor"] = [&]() { m_epsilonFactor = nextFloat(); };
  keywords["lensShader"] = [&]() {
    const int lens = nextInt();
    m_lensShader = (lens < LENS_SHADER_PINHOLE || LENS_SHADER_SPHERE < lens) ? LENS_SHADER_PINHOLE : static_cast<LensShader>(lens);
  };
  keywords["center"] = [&]() { const float x = nextFloat(), y = nextFloat(), z = nextFloat(); m_camera.m_center = make_float3(x, y, z); m_camera.markDirty(); };
  keywords["camera"] = [&]() { m_camera.m_phi = nextFloat(); m_camera.m_theta = nextFloat(); m_camera.m_fov = nextFloat(); m_camera.m_distance = nextFloat(); m_camera.markDirty(); };
  keywords["prefixScreenshot"] = [&]() { parser.getNextLine(token); m_prefixScreenshot = token; };
  keywords["gamma"] = [&]() { m_tonemapperGUI.gamma = nextFloat(); };
  keywords["colorBalance"] = [&]() { for (int i = 0; i < 3; ++i) m_tonemapperGUI.colorBalance[i] = nextFloat(); };
  keywords["whitePoint"] = [&]() { m_tonemapperGUI.whitePoint = nextFloat(); };
  keywords["burnHighlights"] = [&]() { m_tonemapperGUI.burnHighlights = nextFloat(); };
  keywords["crushBlacks"] = [&]() { m_tonemapperGUI.crushBlacks = nextFloat(); };
  keywords["saturation"] = [&]() { m_tonemapperGUI.saturation = nextFloat(); };
  keywords["brightness"] = [&]() { m_tonemapperGUI.brightness = nextFloat(); };
  // extensions of this build (the reference would print its unknown-option warning and carry on)
  keywords["textureAlbedo"] = [&]() { parser.getNextLine(token); m_fileAlbedo = token; };
  keywords["textureCutout"] = [&]() { parser.getNextLine(token); m_fileCutout = token; };
  keywords["composite"] = [&]() { m_compositeMode = nextInt(); };
  keywords["batchIterations"] = [&]() { m_batch = std::max(1, nextInt()); };
  keywords["coalesceIterations"] = [&]() { m_coalesce = std::max(0, nextInt()); };

  while ((tokenType = parser.getNextToken(token)) != PTT_EOF)
  {
    if (tokenType == PTT_UNKNOWN)
    {
      std::cerr << "ERROR: loadSystemDescription() " << filename << " (" << parser.getLine() << "): Unknown token type." << std::endl;
      return false;
    }
    if (tokenType != PTT_ID) continue;
    auto it = keywords.find(token);
    if (it != keywords.end()) it->second();
    else std::cerr << "WARNING: loadSystemDescription(): Unknown system option name: " << token << std::endl;
  }
  return true;
}

// ------------------------------------------------------------------------------------------------------------------
// Scene description (Application.cpp:1397-1878): a state machine over the current material parameters and the
// current transform; `material` snapshots the parameters, `model` instantiates cached procedural geometry.
// ------------------------------------------------------------------------------------------------------------------
void Application::appendInstance(std::shared_ptr<sg::Group>& group, std::shared_ptr<sg::Triangles> geometry, const float trafo[12],
                                 std::string const& reference, unsigned int& idInstance)
{
  std::shared_ptr<sg::Instance> instance(new sg::Instance(idInstance++));
  instance->setTransform(trafo);
  instance->setChild(geometry);
  int indexMaterial = -1;
  std::map<std::string, int>::const_iterator itm = m_mapMaterialReferences.find(reference);
  if (itm != m_mapMaterialReferences.end()) indexMaterial = itm->second;
  else
  {
    std::cerr << "WARNING: loadSceneDescription() No material found for " << reference << ". Trying default." << std::endl;
    std::map<std::string, int>::const_iterator itmd = m_mapMaterialReferences.find(std::string("default"));
    if (itmd != m_mapMaterialReferences.end()) indexMaterial = itmd->second;
    else std::cerr << "ERROR: loadSceneDescription() No default material found" << std::endl;
  }
  instance->setMaterial(indexMaterial);
  group->addChild(instance);
}

std::shared_ptr<sg::Triangles> Application::cachedGeometry(std::string const& key, bool& created)
{
  std::map<std::string, unsigned int>::const_iterator it = m_mapGeometries.find(key);
  created = (it == m_mapGeometries.end());
  if (!created) return m_geometries[it->second];
  m_mapGeometries[key] = m_idGeometry;
  std::shared_ptr<sg::Triangles> geometry = std::make_shared<sg::Triangles>(m_idGeometry++);
  m_geometries.push_back(geometry);
  return geometry;
}

bool Application::loadSceneDescription(std::string const& filename)
{
  Parser parser;
  if (!parser.load(filename)) return false;

  std::string token;
  ParserTokenType tokenType;
  auto nextInt = [&]() { parser.getNextToken(token); return std::atoi(token.c_str()); };
  auto nextFloat = [&]() { parser.getNextToken(token); return (float)std::atof(token.c_str()); };

  std::stack<Mat44> stackMatrix;
  Mat44 curMatrix = Mat44::identity();   // object to world, row-vector convention

  float3 curAlbedo = make_float3(1.0f);
  float2 curRoughness = make_float2(0.1f, 0.1f);
  float3 curAbsorptionColor = make_float3(1.0f);
  float  curAbsorptionScale = 0.0f;
  float  curIOR = 1.5f;
  bool   curThinwalled = false;
  bool   curAlbedoTexture = false, curCutoutTexture = false;   // extension keywords: the reference sets these from the GUI only

  static const std::map<std::string, FunctionIndex> bsdfNames = {
    { "brdf_diffuse", INDEX_BRDF_DIFFUSE }, { "brdf_specular", INDEX_BRDF_SPECULAR }, { "bsdf_specular", INDEX_BSDF_SPECULAR },
    { "brdf_ggx_smith", INDEX_BRDF_GGX_SMITH }, { "bsdf_ggx_smith", INDEX_BSDF_GGX_SMITH } };

  while ((tokenType = parser.getNextToken(token)) != PTT_EOF)
  {
    if (tokenType == PTT_UNKNOWN)
    {
      std::cerr << "ERROR: loadSceneDescription() " << filename << " (" << parser.getLine() << "): Unknown token type." << std::endl;
      return false;
    }
    if (tokenType != PTT_ID) continue;

    if (token == "albedo") { curAlbedo.x = nextFloat(); curAlbedo.y = nextFloat(); curAlbedo.z = nextFloat(); }
    else if (token == "roughness") { curRoughness.x = nextFloat(); curRoughness.y = nextFloat(); }
    else if (token == "absorption") { curAbsorptionColor.x = nextFloat(); curAbsorptionColor.y = nextFloat(); curAbsorptionColor.z = nextFloat(); }
    else if (token == "absorptionScale") { curAbsorptionScale = nextFloat(); }
    else if (token == "ior") { curIOR = nextFloat(); }
    else if (token == "thinwalled") { curThinwalled = (nextInt() != 0); }
    else if (token == "albedoTexture") { curAlbedoTexture = (nextInt() != 0); }
    else if (token == "cutoutTexture") { curCutoutTexture = (nextInt() != 0); }
    else if (token == "material")
    {
      std::string nameMaterialReference, nameMaterial;
      parser.getNextToken(nameMaterialReference);   // duplicates: the last definition wins the name
      parser.getNextToken(nameMaterial);
      const int indexMaterial = static_cast<int>(m_materialsGUI.size());
      MaterialGUI materialGUI;
      materialGUI.name = nameMaterialReference;
      materialGUI.indexBSDF = INDEX_BRDF_DIFFUSE;
      std::map<std::string, FunctionIndex>::const_iterator itb = bsdfNames.find(nameMaterial);
      if (itb != bsdfNames.end()) materialGUI.indexBSDF = itb->second;
      else std::cerr << "WARNING: loadSceneDescription() unknown material " << nameMaterial << std::endl;
      materialGUI.albedo = curAlbedo;
      materialGUI.roughness = curRoughness;
      materialGUI.absorptionColor = curAbsorptionColor;
      materialGUI.absorptionScale = curAbsorptionScale;
      materialGUI.ior = curIOR;
      materialGUI.thinwalled = curThinwalled;
      materialGUI.useAlbedoTexture = curAlbedoTexture;
      materialGUI.useCutoutTexture = curCutoutTexture;
      m_materialsGUI.push_back(materialGUI);
      m_mapMaterialReferences[nameMaterialReference] = indexMaterial;
    }
    else if (token == "identity") { curMatrix = Mat44::identity(); }
    else if (token == "push") { stackMatrix.push(curMatrix); }
    else if (token == "pop")
    {
      if (!stackMatrix.empty()) { curMatrix = stackMatrix.top(); stackMatrix.pop(); }
      else { std::cerr << "ERROR: loadSceneDescription() pop on empty stack. Resetting to identity." << std::endl; curMatrix = Mat44::identity(); }
    }
    else if (token == "rotate")
    {
      float axis[3] = { nextFloat(), 0.0f, 0.0f };
      axis[1] = nextFloat(); axis[2] = nextFloat();
      const float len = std::sqrt(axis[0] * axis[0] + axis[1] * axis[1] + axis[2] * axis[2]);
      for (int k = 0; k < 3; ++k) axis[k] /= len;
      const float degrees = nextFloat();
      const float angle = degrees * (RT_PI_F / 180.0f);
      curMatrix = curMatrix * Mat44::rotation(axis, angle);
    }
    else if (token == "scale") { const float x = nextFloat(), y = nextFloat(), z = nextFloat(); curMatrix = curMatrix * Mat44::scaling(x, y, z); }
    else if (token == "translate") { const float x = nextFloat(), y = nextFloat(), z = nextFloat(); curMatrix = curMatrix * Mat44::translation(x, y, z); }
    else if (token == "model")
    {
      parser.getNextToken(token);
      float trafo[12];
      curMatrix.toTrafo(trafo);
      bool created = false;
      if (token == "plane")
      {
        const unsigned int tessU = (unsigned int)nextInt(), tessV = (unsigned int)nextInt(), upAxis = (unsigned int)nextInt();
        std::string ref; parser.getNextToken(ref);
        std::ostringstream key; key << "plane_" << tessU << "_" << tessV << "_" << upAxis;
        std::shared_ptr<sg::Triangles> geometry = cachedGeometry(key.str(), created);
        if (created) geometry->createPlane(tessU, tessV, upAxis);
        appendInstance(m_scene, geometry, trafo, ref, m_idInstance);
      }
      else if (token == "box")
      {
        std::string ref; parser.getNextToken(ref);
        std::shared_ptr<sg::Triangles> geometry = cachedGeometry("box_1_1", created);
        if (created) geometry->createBox();
        appendInstance(m_scene, geometry, trafo, ref, m_idInstance);
      }
      else if (token == "sphere")
      {
        const unsigned int tessU = (unsigned int)nextInt(), tessV = (unsigned int)nextInt();
        const float theta = nextFloat();   // [0, 1]: 1 = closed sphere, smaller values open the north pole
        std::string ref; parser.getNextToken(ref);
        std::ostringstream key; key << "sphere_" << tessU << "_" << tessV << "_" << theta;
        std::shared_ptr<sg::Triangles> geometry = cachedGeometry(key.str(), created);
        if (created) geometry->createSphere(tessU, tessV, 1.0f, theta * RT_PI_F);
        appendInstance(m_scene, geometry, trafo, ref, m_idInstance);
      }
      else if (token == "torus")
      {
        const unsigned int tessU = (unsigned int)nextInt(), tessV = (unsigned int)nextInt();
        const float innerRadius = nextFloat(), outerRadius = nextFloat();
        std::string ref; parser.getNextToken(ref);
        std::ostringstream key; key << "torus_" << tessU << "_" << tessV << "_" << innerRadius << "_" << outerRadius;
        std::shared_ptr<sg::Triangles> geometry = cachedGeometry(key.str(), created);
        if (created) geometry->createTorus(tessU, tessV, innerRadius, outerRadius);
        appendInstance(m_scene, geometry, trafo, ref, m_idInstance);
      }
      else if (token == "assimp")
      {
        std::string filenameModel;
        parser.getNextLine(filenameModel);
        // relative model paths are tried as given and then next to the scene file
        if (!filenameModel.empty() && filenameModel[0] != '/')
        {
          FILE* probe = std::fopen(filenameModel.c_str(), "rb");
          if (probe) std::fclose(probe);
          else
          {
            const size_t slash = filename.find_last_of("/\\");
            if (slash != std::string::npos) filenameModel = filename.substr(0, slash + 1) + filenameModel;
          }
        }
        std::shared_ptr<sg::Group> model = createASSIMP(filenameModel);
        std::shared_ptr<sg::Instance> instance(new sg::Instance(m_idInstance++));
        instance->setTransform(trafo);
        instance->setChild(model);
        m_scene->addChild(instance);
      }
      else std::cerr << "WARNING: loadSceneDescription() unknown model type " << token << std::endl;
    }
    else std::cerr << "loadSceneDescription(): Unknown token " << token << " ignored." << std::endl;
  }
  std::cout << "loadSceneDescription(): m_idGroup = " << m_idGroup << ", m_idInstance = " << m_idInstance << ", m_idGeometry = " << m_idGeometry << std::endl;
  return true;
}

// Same walk as Device::traverseNode, recorded on the host so tools can hand the identical scene to a checker.
void Application::flatten(std::shared_ptr<sg::Node> node, const float matrix[12], int material, int light)
{
  switch (node->getType())
  {
    case sg::NT_GROUP:
    {
      std::shared_ptr<sg::Group> group = std::dynamic_pointer_cast<sg::Group>(node);
      for (size_t i = 0; i < group->getNumChildren(); ++i) flatten(group->getChild(i), matrix, material, light);
      break;
    }
    case sg::NT_INSTANCE:
    {
      std::shared_ptr<sg::Instance> instance = std::dynamic_pointer_cast<sg::Instance>(node);
      float trafo[12];
      multiplyMatrix(trafo, matrix, instance->getTransform());
      if (0 <= instance->getMaterial()) material = instance->getMaterial();
      if (0 <= instance->getLight()) light = instance->getLight();
      if (instance->getChild()) flatten(instance->getChild(), trafo, material, light);
      break;
    }
    case sg::NT_TRIANGLES:
    {
      FlatInstance fi;
      std::memcpy(fi.transform, matrix, sizeof(float) * 12);
      fi.geometry = (int)node->getId(); fi.material = material; fi.light = light;
      m_flatInstances.push_back(fi);
      break;
    }
  }
}
