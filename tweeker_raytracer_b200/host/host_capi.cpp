// host_capi.cpp -- flat C entry points over the C++ host classes, for tools and the Python test harness
// (ctypes).  Nothing here computes pixels: rendering goes Application -> Raytracer -> Device -> librtcore.
#include <cstring>
#include <string>

#include "Application.h"

extern "C" {

struct rth_info
{
  int resolutionX, resolutionY, samplesSqrt, miss, lightMode, strategy, numDevices;
  int numGeometries, numInstances, numMaterials, numLights, hasEnvironment;
};

static std::string g_error;
const char* rth_last_error(void) { return g_error.c_str(); }

void* rth_app_create(const char* systemFile, const char* sceneFile, int hostOnly)
{
  Options options;
  options.set(512, 512, 1, systemFile ? systemFile : "", sceneFile ? sceneFile : "");
  Application* app = nullptr;
  try { app = new Application(options, hostOnly != 0); }
  catch (std::exception const& e) { g_error = e.what(); return nullptr; }
  if (!app->isValid()) { g_error = app->getLastError(); delete app; return nullptr; }
  return app;
}

void rth_app_destroy(void* h) { delete static_cast<Application*>(h); }

int rth_app_info(void* h, rth_info* out)
{
  Application* app = static_cast<Application*>(h);
  std::memset(out, 0, sizeof(*out));
  out->resolutionX = app->getResolution().x; out->resolutionY = app->getResolution().y;
  out->samplesSqrt = app->getState().samplesSqrt; out->miss = app->getMiss(); out->lightMode = app->getLightMode();
  out->strategy = (int)app->getStrategy();
  out->numDevices = app->getRaytracer() ? (int)app->getRaytracer()->m_activeDevices.size() : 0;
  out->numGeometries = (int)app->getGeometries().size(); out->numInstances = (int)app->getFlatInstances().size();
  out->numMaterials = (int)app->getMaterialsGUI().size(); out->numLights = (int)app->getLights().size();
  out->hasEnvironment = app->getEnvironment() && app->getEnvironment()->getWidth() ? 1 : 0;
  return 0;
}

int rth_app_geometry(void* h, int g, const rt_TriangleAttributes** attrs, unsigned int* numVerts, const unsigned int** indices, unsigned int* numTris)
{
  Application* app = static_cast<Application*>(h);
  if (g < 0 || (size_t)g >= app->getGeometries().size()) return -1;
  sg::Triangles const& t = *app->getGeometries()[g];
  *attrs = t.getAttributes().data(); *numVerts = (unsigned int)t.getAttributes().size();
  *indices = t.getIndices().data(); *numTris = (unsigned int)(t.getIndices().size() / 3);
  return 0;
}

int rth_app_instance(void* h, int i, float transform[12], int* geometry, int* material, int* light)
{
  Application* app = static_cast<Application*>(h);
  if (i < 0 || (size_t)i >= app->getFlatInstances().size()) return -1;
  FlatInstance const& fi = app->getFlatInstances()[i];
  std::memcpy(transform, fi.transform, sizeof(float) * 12);
  *geometry = fi.geometry; *material = fi.material; *light = fi.light;
  return 0;
}

int rth_app_materials(void* h, rt_MaterialDefinition* out)
{
  std::vector<MaterialDefinition> m;
  static_cast<Application*>(h)->getMaterialDefinitions(m);
  std::memcpy(out, m.data(), m.size() * sizeof(MaterialDefinition));
  return (int)m.size();
}

int rth_app_lights(void* h, rt_LightDefinition* out)
{
  std::vector<LightDefinition> const& l = static_cast<Application*>(h)->getLights();
  if (!l.empty()) std::memcpy(out, l.data(), l.size() * sizeof(LightDefinition));
  return (int)l.size();
}

int rth_app_camera(void* h, rt_CameraDefinition* out) { *out = static_cast<Application*>(h)->getCameras()[0]; return 0; }

int rth_app_system_data(void* h, int deviceIndex, rt_SystemData* out) { static_cast<Application*>(h)->getSystemData(deviceIndex, *out); return 0; }

int rth_app_tonemapper(void* h, rt_TonemapperParams* out) { *out = static_cast<Application*>(h)->getTonemapper(); return 0; }

int rth_app_environment(void* h, unsigned int* w, unsigned int* hgt, const float** texels, const float** cdfU, const float** cdfV, float* integral)
{
  EnvMap const* env = static_cast<Application*>(h)->getEnvironment();
  if (!env || env->getWidth() == 0) return -1;
  *w = env->getWidth(); *hgt = env->getHeight(); *texels = env->getTexels().data();
  *cdfU = env->getCDF_U().data(); *cdfV = env->getCDF_V().data(); *integral = env->getIntegral();
  return 0;
}

int rth_app_save_system(void* h, const char* filename, char* path, int pathLen)
{
  std::string written;
  const bool ok = static_cast<Application*>(h)->saveSystemDescription(filename ? filename : "", &written);
  if (path && pathLen > 0) std::snprintf(path, (size_t)pathLen, "%s", written.c_str());
  return ok ? 0 : -1;
}

// mutators (valid in host-only mode too: they update the host scene; with devices they also restart the accumulation)
void rth_app_set_camera(void* h, float phi, float theta, float fov, float distance, const float center[3])
{
  static_cast<Application*>(h)->setCamera(phi, theta, fov, distance, center);
}

int rth_app_update_material(void* h, int index, int indexBSDF, const float albedo[3], const float roughness[2], const float absorptionColor[3],
                            float absorptionScale, float ior, int thinwalled)
{
  Application* app = static_cast<Application*>(h);
  MaterialGUI m;
  if (0 <= index && (size_t)index < app->getMaterialsGUI().size())      // the texture check boxes keep their state
  { m.useAlbedoTexture = app->getMaterialsGUI()[index].useAlbedoTexture; m.useCutoutTexture = app->getMaterialsGUI()[index].useCutoutTexture; }
  m.indexBSDF = static_cast<FunctionIndex>(indexBSDF);
  m.albedo = make_float3(albedo[0], albedo[1], albedo[2]);
  m.roughness = make_float2(roughness[0], roughness[1]);
  m.absorptionColor = make_float3(absorptionColor[0], absorptionColor[1], absorptionColor[2]);
  m.absorptionScale = absorptionScale; m.ior = ior; m.thinwalled = thinwalled != 0;
  try { return static_cast<Application*>(h)->updateMaterial(index, m) ? 0 : -1; } catch (std::exception const& e) { g_error = e.what(); return -2; }
}

// the GUI's "use albedo texture" / "use cutout texture" check boxes of one material (MaterialGUI.h:47-48)
int rth_app_update_material_textures(void* h, int index, int useAlbedo, int useCutout)
{
  Application* app = static_cast<Application*>(h);
  if (index < 0 || (size_t)index >= app->getMaterialsGUI().size()) return -1;
  MaterialGUI m = app->getMaterialsGUI()[index];
  m.useAlbedoTexture = useAlbedo != 0; m.useCutoutTexture = useCutout != 0;
  try { return app->updateMaterial(index, m) ? 0 : -1; } catch (std::exception const& e) { g_error = e.what(); return -2; }
}

// the material pictures: name = "albedo" | "cutout"; texels = RGBA32F, row 0 = v 0
int rth_app_picture(void* h, const char* name, unsigned int* w, unsigned int* hgt, const float** texels)
{
  EnvMap* p = static_cast<Application*>(h)->getPicture(name ? name : "");
  if (!p || p->getWidth() == 0) return -1;
  *w = p->getWidth(); *hgt = p->getHeight(); *texels = p->getTexels().data();
  return 0;
}

int rth_app_update_light_emission(void* h, int index, const float emission[3])
{
  try { return static_cast<Application*>(h)->updateLightEmission(index, emission) ? 0 : -1; } catch (std::exception const& e) { g_error = e.what(); return -2; }
}

// instance `index` in the numbering of rth_app_instance; matrix: object -> world, row-major 3x4
int rth_app_update_instance_transform(void* h, int index, const float matrix[12])
{
  try { return static_cast<Application*>(h)->updateInstanceTransform(index, matrix) ? 0 : -1; } catch (std::exception const& e) { g_error = e.what(); return -2; }
}

// a new instance-level topology on every device (after large motion); frames do not change
int rth_app_rebuild_instance_level(void* h)
{
  try { static_cast<Application*>(h)->rebuildInstanceLevel(); return 0; } catch (std::exception const& e) { g_error = e.what(); return -2; }
}

// new vertex records (48 B each, numVerts = the geometry's) of geometry `g` in the numbering of rth_app_geometry; rebuild != 0: a
// new GAS topology (after large deformation) instead of a refit
int rth_app_update_geometry(void* h, int g, const rt_TriangleAttributes* attributes, unsigned int numVerts, int rebuild)
{
  try
  {
    return static_cast<Application*>(h)->updateGeometry(g, reinterpret_cast<const TriangleAttributes*>(attributes), numVerts, rebuild != 0) ? 0 : -1;
  }
  catch (std::exception const& e) { g_error = e.what(); return -2; }
}

// --- device side (needs a GPU) ---
unsigned int rth_app_render(void* h, unsigned int count) { return static_cast<Application*>(h)->render(count); }
// the reference's calling pattern: `calls` times the unchanged `unsigned int Raytracer::render()` (one iteration per call)
unsigned int rth_app_render_calls(void* h, unsigned int calls)
{
  Raytracer* rt = static_cast<Application*>(h)->getRaytracer();
  unsigned int it = 0;
  try { for (unsigned int k = 0; k < calls; ++k) it = rt->render(); } catch (std::exception const& e) { g_error = e.what(); }
  return it;
}
// Raytracer::setCoalesceLimit (1 = every render() launches); returns the previous limit
unsigned int rth_app_set_coalesce(void* h, unsigned int limit)
{
  Raytracer* rt = static_cast<Application*>(h)->getRaytracer();
  const unsigned int before = rt->getCoalesceLimit();
  try { rt->setCoalesceLimit(limit); } catch (std::exception const& e) { g_error = e.what(); }
  return before;
}
int rth_app_synchronize(void* h)
{
  try { static_cast<Application*>(h)->getRaytracer()->synchronize(); return 0; } catch (std::exception const& e) { g_error = e.what(); return -1; }
}
const float* rth_app_frame(void* h) { return static_cast<Application*>(h)->getOutputBufferHost(); }
// a rank's own running average (no collective); the same as rth_app_frame outside a process group
const float* rth_app_local_frame(void* h)
{
  try { return reinterpret_cast<const float*>(static_cast<Application*>(h)->getRaytracer()->getLocalOutputBufferHost()); }
  catch (std::exception const& e) { g_error = e.what(); return nullptr; }
}
void rth_app_restart(void* h) { static_cast<Application*>(h)->restartAccumulation(); }
void rth_app_set_composite(void* h, int mode) { static_cast<Application*>(h)->setCompositeMode(mode); }
double rth_app_benchmark(void* h) { Application* app = static_cast<Application*>(h); app->benchmark(); return app->getLastBenchmarkSeconds(); }
int rth_app_screenshot(void* h, int tonemap, char* path, int pathLen)
{
  std::string written;
  const bool ok = static_cast<Application*>(h)->screenshot(tonemap != 0, &written);
  if (path && pathLen > 0) std::snprintf(path, (size_t)pathLen, "%s", written.c_str());
  return ok ? 0 : -1;
}
int rth_app_tonemap(void* h, unsigned char* rgb)
{
  try { std::vector<unsigned char> v; static_cast<Application*>(h)->tonemapDevice(v); std::memcpy(rgb, v.data(), v.size()); return 0; }
  catch (std::exception const& e) { g_error = e.what(); return -1; }
}
rtc_context* rth_app_context(void* h, int deviceIndex)
{
  Raytracer* rt = static_cast<Application*>(h)->getRaytracer();
  if (!rt || deviceIndex < 0 || (size_t)deviceIndex >= rt->m_activeDevices.size()) return nullptr;
  return rt->m_activeDevices[deviceIndex]->getContext();
}
// --- one process per GPU: sample-range partition + NCCL mean of the frames (Raytracer::joinProcessGroup) ---
int rth_process_group_id(char id[128])
{
  try { Application::makeProcessGroupId(id); return 0; } catch (std::exception const& e) { g_error = e.what(); return -1; }
}
int rth_app_join_group(void* h, int rank, int world, const char id[128])
{
  Application* app = static_cast<Application*>(h);
  if (!app->getRaytracer()) { g_error = "host-only Application has no Raytracer"; return -2; }
  if (!app->joinProcessGroup(rank, world, id)) { g_error = app->getLastError(); return -1; }
  return 0;
}
int rth_app_group_reduce_mean(void* h, uint64_t src, uint64_t dst, uint64_t count)
{
  try { static_cast<Application*>(h)->getRaytracer()->reduceMeanToRoot(src, dst, (size_t)count); return 0; }
  catch (std::exception const& e) { g_error = e.what(); return -1; }
}
// pure index arithmetic (no device): the iteration range rank `rank` of `world` renders out of samplesPerPixel
void rth_sample_range(unsigned int samplesPerPixel, int rank, int world, unsigned int* first, unsigned int* count)
{
  *count = Raytracer::samplesPerRank(samplesPerPixel, world);
  *first = (1 < world) ? (unsigned int)rank * *count : 0u;
}
int rth_app_stats(void* h, rtc_stats* out)
{
  try { static_cast<Application*>(h)->getRaytracer()->getStats(*out); return 0; } catch (std::exception const& e) { g_error = e.what(); return -1; }
}

} // extern "C"
