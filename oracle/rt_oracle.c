/*
 * rt_oracle.c -- TEST INFRASTRUCTURE ONLY (see rt_oracle.h).  Scalar CPU restatement of the
 * rtigo3 hot path in plain C.  Nothing under tweeker_raytracer_b200/ links or calls this file.
 *
 * Build: gcc -O2 -ffp-contract=off -mfma (explicit fmaf() only where the arithmetic is DEFINED
 * with a fused multiply-add; the compiler never contracts on its own).
 *
 * Paths are relative to /root/reference/apps/rtigo3/.
 */
#define _GNU_SOURCE
#include "rt_oracle.h"
#include "rt_portable_math.h"

#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

/* ------------------------------------------------------------------------------------------
 * small vector layer; every operation is component-wise in the order vector_math.h uses
 * (shaders/vector_math.h:574-608: dot = x*x' + y*y' + z*z'; normalize = v * (1/sqrt(dot));
 * v / s = v * (1/s), :530-534; reflect = i - 2*n*dot(n,i), :605-608; lerp = a + t*(b-a), :547)
 * ------------------------------------------------------------------------------------------ */
typedef struct { float x, y, z; } v3;
typedef struct { float x, y; } v2;
typedef struct { float x, y, z, w; } v4;

static inline v3 V3(float x, float y, float z) { v3 r = { x, y, z }; return r; }
static inline v3 v3s(float s) { return V3(s, s, s); }
static inline v3 vadd(v3 a, v3 b) { return V3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 vsub(v3 a, v3 b) { return V3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 vmul(v3 a, v3 b) { return V3(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 vscale(v3 a, float s) { return V3(a.x * s, a.y * s, a.z * s); }
static inline v3 vneg(v3 a) { return V3(-a.x, -a.y, -a.z); }
static inline float vdot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline v3 vcross(v3 a, v3 b) { return V3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
static inline float vlength(v3 a) { return sqrtf(vdot(a, a)); }
static inline v3 vnormalize(v3 a) { const float inv = 1.0f / sqrtf(vdot(a, a)); return vscale(a, inv); }
static inline v3 vdivs(v3 a, float s) { const float inv = 1.0f / s; return vscale(a, inv); }
static inline v3 vreflect(v3 i, v3 n) { return vsub(i, vscale(vscale(n, 2.0f), vdot(n, i))); }
static inline int v3_is_null(v3 v) { return v.x == 0.0f && v.y == 0.0f && v.z == 0.0f; }
static inline v3 from_f3(rt_float3 f) { return V3(f.x, f.y, f.z); }
static inline float fmax3(v3 a) { return fmaxf(fmaxf(a.x, a.y), a.z); }

/* shader_common.h:157-187 */
static inline float intensity3(v3 c) { return (c.x + c.y + c.z) * 0.3333333333f; }
static inline float power_heuristic(float a, float b) { const float t = a * a; return t / (t + b * b); }

/* ------------------------------------------------------------------------------------------
 * RNG  (shaders/random_number_generators.h:39-78)
 * ------------------------------------------------------------------------------------------ */
uint32_t orc_tea4(uint32_t v0, uint32_t v1)
{
  uint32_t s0 = 0;
  for (int n = 0; n < 4; ++n)
  {
    s0 += 0x9e3779b9u;
    v0 += ((v1 << 4) + 0xA341316Cu) ^ (v1 + s0) ^ ((v1 >> 5) + 0xC8013EA4u);
    v1 += ((v0 << 4) + 0xAD90777Du) ^ (v0 + s0) ^ ((v0 >> 5) + 0x7E95761Eu);
  }
  return v0;
}

float orc_rng(uint32_t* state)
{
  *state = *state * 1664525u + 1013904223u;
  return (float)(*state & 0x00FFFFFFu) / (float)0x01000000u;
}

static inline v2 rng2(uint32_t* state)
{
  v2 s;
  s.x = orc_rng(state);
  s.y = orc_rng(state);
  return s;
}

int orc_uses_libm(void)
{
#ifdef RT_MATH_LIBM
  return 1;
#else
  return 0;
#endif
}

int orc_online_cores(void)
{
  long n = sysconf(_SC_NPROCESSORS_ONLN);
  return n < 1 ? 1 : (int)n;
}

/* ------------------------------------------------------------------------------------------
 * Scene
 * ------------------------------------------------------------------------------------------ */
typedef struct { float lo[3], hi[3]; } aabb;

typedef struct {
  aabb     box;
  uint32_t left;    /* inner: index of left child (right = left + 1); leaf: first primitive slot */
  uint32_t count;   /* 0 = inner, else number of primitives */
} bnode;

typedef struct {
  bnode*    nodes;
  uint32_t  numNodes;
  uint32_t* prims;   /* permutation of primitive ids */
} bvh;

typedef struct {
  rt_TriangleAttributes* attrs;
  uint32_t  numVerts;
  uint32_t* indices;
  uint32_t  numTris;
  bvh       tree;
  aabb      bounds;
} geometry;

typedef struct {
  float m[12];     /* object -> world, row-major 3x4 */
  float inv[12];   /* world -> object */
  int   geometry;
  int   material;
  int   light;
  aabb  world;
  int   active;    /* 0: inactive (tri_active's comment): no ray hits the instance */
} instance;

struct orc_scene {
  geometry* geoms;   int numGeoms,   capGeoms;
  instance* insts;   int numInsts,   capInsts;
  rt_MaterialDefinition* materials;  int numMaterials;
  rt_LightDefinition*    lights;     int numLightDefs;
  rt_CameraDefinition    camera;
  float*   envTexels; uint32_t envW, envH;
  float*   envCdfU;   float* envCdfV; float envIntegral;
  bvh      top;
  int      committed;
  int      hasCutout;   /* some material carries a cutout texture: traces take the ordered any-hit path */
};

orc_scene* orc_scene_create(void) { return (orc_scene*)calloc(1, sizeof(orc_scene)); }

static void bvh_free(bvh* b) { free(b->nodes); free(b->prims); memset(b, 0, sizeof(*b)); }

void orc_scene_destroy(orc_scene* s)
{
  if (!s) return;
  for (int i = 0; i < s->numGeoms; ++i)
  {
    free(s->geoms[i].attrs);
    free(s->geoms[i].indices);
    bvh_free(&s->geoms[i].tree);
  }
  free(s->geoms); free(s->insts); free(s->materials); free(s->lights);
  free(s->envTexels); free(s->envCdfU); free(s->envCdfV);
  bvh_free(&s->top);
  free(s);
}

int orc_scene_add_geometry(orc_scene* s, const rt_TriangleAttributes* attrs, uint32_t numVerts,
                           const uint32_t* indices, uint32_t numTris)
{
  if (s->numGeoms == s->capGeoms)
  {
    s->capGeoms = s->capGeoms ? 2 * s->capGeoms : 8;
    s->geoms = (geometry*)realloc(s->geoms, sizeof(geometry) * (size_t)s->capGeoms);
  }
  geometry* g = &s->geoms[s->numGeoms];
  memset(g, 0, sizeof(*g));
  g->attrs = (rt_TriangleAttributes*)malloc(sizeof(rt_TriangleAttributes) * (size_t)numVerts);
  memcpy(g->attrs, attrs, sizeof(rt_TriangleAttributes) * (size_t)numVerts);
  g->indices = (uint32_t*)malloc(sizeof(uint32_t) * 3u * (size_t)numTris);
  memcpy(g->indices, indices, sizeof(uint32_t) * 3u * (size_t)numTris);
  g->numVerts = numVerts;
  g->numTris = numTris;
  return s->numGeoms++;
}

int orc_scene_add_instance(orc_scene* s, const float transform[12], int geom, int material, int light)
{
  if (s->numInsts == s->capInsts)
  {
    s->capInsts = s->capInsts ? 2 * s->capInsts : 8;
    s->insts = (instance*)realloc(s->insts, sizeof(instance) * (size_t)s->capInsts);
  }
  instance* in = &s->insts[s->numInsts];
  memset(in, 0, sizeof(*in));
  memcpy(in->m, transform, sizeof(float) * 12);
  in->geometry = geom; in->material = material; in->light = light;
  return s->numInsts++;
}

void orc_scene_set_materials(orc_scene* s, const rt_MaterialDefinition* m, int n)
{
  free(s->materials);
  s->materials = (rt_MaterialDefinition*)malloc(sizeof(*m) * (size_t)(n > 0 ? n : 1));
  memcpy(s->materials, m, sizeof(*m) * (size_t)n);
  s->numMaterials = n;
  s->hasCutout = 0;
  for (int i = 0; i < n; ++i) if (m[i].textureCutout != 0) s->hasCutout = 1;
}

void orc_scene_set_lights(orc_scene* s, const rt_LightDefinition* l, int n)
{
  free(s->lights);
  s->lights = (rt_LightDefinition*)malloc(sizeof(*l) * (size_t)(n > 0 ? n : 1));
  if (n > 0) memcpy(s->lights, l, sizeof(*l) * (size_t)n);
  s->numLightDefs = n;
}

void orc_scene_set_camera(orc_scene* s, const rt_CameraDefinition* c) { s->camera = *c; }

void orc_scene_set_env(orc_scene* s, const float* rgba, uint32_t w, uint32_t h,
                       const float* cdfU, const float* cdfV, float integral)
{
  free(s->envTexels); free(s->envCdfU); free(s->envCdfV);
  s->envTexels = (float*)malloc(sizeof(float) * 4u * (size_t)w * h);
  memcpy(s->envTexels, rgba, sizeof(float) * 4u * (size_t)w * h);
  s->envCdfU = (float*)malloc(sizeof(float) * (size_t)(w + 1) * h);
  memcpy(s->envCdfU, cdfU, sizeof(float) * (size_t)(w + 1) * h);
  s->envCdfV = (float*)malloc(sizeof(float) * (size_t)(h + 1));
  memcpy(s->envCdfV, cdfV, sizeof(float) * (size_t)(h + 1));
  s->envW = w; s->envH = h; s->envIntegral = integral;
}

/* ------------------------------------------------------------------------------------------
 * The instance inverse (DEFINED here; OptiX computed it inside optixAccelBuild, src/Device.cpp:1478,
 * read back through optixGetInstanceInverseTransformFromHandle, shaders/closesthit.cu:49-52).
 * Adjugate / determinant of the upper 3x3 in double, rounded once to float; translation
 * -(Minv * t) in double.  The core uses the same definition (csrc/rtc_scene.cpp).
 * ------------------------------------------------------------------------------------------ */
static void invert_3x4(const float m[12], float out[12])
{
  const double a = m[0], b = m[1], c = m[2],  tx = m[3];
  const double d = m[4], e = m[5], f = m[6],  ty = m[7];
  const double g = m[8], h = m[9], i = m[10], tz = m[11];
  const double c00 = e * i - f * h, c01 = c * h - b * i, c02 = b * f - c * e;
  const double c10 = f * g - d * i, c11 = a * i - c * g, c12 = c * d - a * f;
  const double c20 = d * h - e * g, c21 = b * g - a * h, c22 = a * e - b * d;
  const double det = a * c00 + b * c10 + c * c20;
  const double r = 1.0 / det;
  const double i00 = c00 * r, i01 = c01 * r, i02 = c02 * r;
  const double i10 = c10 * r, i11 = c11 * r, i12 = c12 * r;
  const double i20 = c20 * r, i21 = c21 * r, i22 = c22 * r;
  out[0] = (float)i00; out[1] = (float)i01; out[2]  = (float)i02; out[3]  = (float)(-(i00 * tx + i01 * ty + i02 * tz));
  out[4] = (float)i10; out[5] = (float)i11; out[6]  = (float)i12; out[7]  = (float)(-(i10 * tx + i11 * ty + i12 * tz));
  out[8] = (float)i20; out[9] = (float)i21; out[10] = (float)i22; out[11] = (float)(-(i20 * tx + i21 * ty + i22 * tz));
}

/* ------------------------------------------------------------------------------------------
 * Oracle BVH: a plain binary tree with binned-SAH splits.  Its only job is to make the oracle
 * fast enough; the brute-force mode is the ground truth it is tested against.
 * ------------------------------------------------------------------------------------------ */
static inline void box_empty(aabb* b) { for (int k = 0; k < 3; ++k) { b->lo[k] = INFINITY; b->hi[k] = -INFINITY; } }
static inline void box_grow(aabb* b, const aabb* o)
{
  for (int k = 0; k < 3; ++k) { if (o->lo[k] < b->lo[k]) b->lo[k] = o->lo[k]; if (o->hi[k] > b->hi[k]) b->hi[k] = o->hi[k]; }
}
static inline float box_half_area(const aabb* b)
{
  const float dx = b->hi[0] - b->lo[0], dy = b->hi[1] - b->lo[1], dz = b->hi[2] - b->lo[2];
  return dx * dy + dy * dz + dz * dx;
}

#define ORC_BINS 16
#define ORC_LEAF 4

typedef struct { bvh* tree; const aabb* pb; uint32_t capNodes; } build_ctx;

static void build_rec(build_ctx* c, uint32_t nodeIdx, uint32_t first, uint32_t count)
{
  bvh* t = c->tree;
  aabb box, cbox;
  box_empty(&box); box_empty(&cbox);
  for (uint32_t i = first; i < first + count; ++i)
  {
    const aabb* p = &c->pb[t->prims[i]];
    box_grow(&box, p);
    for (int k = 0; k < 3; ++k)
    {
      const float ce = 0.5f * (p->lo[k] + p->hi[k]);
      if (ce < cbox.lo[k]) cbox.lo[k] = ce;
      if (ce > cbox.hi[k]) cbox.hi[k] = ce;
    }
  }
  t->nodes[nodeIdx].box = box;
  if (count <= ORC_LEAF)
  {
    t->nodes[nodeIdx].left = first; t->nodes[nodeIdx].count = count;
    return;
  }
  int bestAxis = -1, bestSplit = 0; float bestCost = INFINITY;
  for (int axis = 0; axis < 3; ++axis)
  {
    const float ext = cbox.hi[axis] - cbox.lo[axis];
    if (!(ext > 0.0f)) continue;
    aabb bb[ORC_BINS]; uint32_t bc[ORC_BINS];
    for (int b = 0; b < ORC_BINS; ++b) { box_empty(&bb[b]); bc[b] = 0; }
    const float scale = (float)ORC_BINS / ext;
    for (uint32_t i = first; i < first + count; ++i)
    {
      const aabb* p = &c->pb[t->prims[i]];
      int b = (int)((0.5f * (p->lo[axis] + p->hi[axis]) - cbox.lo[axis]) * scale);
      if (b < 0) b = 0; if (b >= ORC_BINS) b = ORC_BINS - 1;
      box_grow(&bb[b], p); bc[b]++;
    }
    float rightArea[ORC_BINS]; aabb acc; box_empty(&acc); uint32_t rc[ORC_BINS]; uint32_t n = 0;
    for (int b = ORC_BINS - 1; b > 0; --b) { box_grow(&acc, &bb[b]); n += bc[b]; rightArea[b] = box_half_area(&acc); rc[b] = n; }
    box_empty(&acc); n = 0;
    for (int b = 0; b < ORC_BINS - 1; ++b)
    {
      box_grow(&acc, &bb[b]); n += bc[b];
      if (n == 0 || rc[b + 1] == 0) continue;
      const float cost = box_half_area(&acc) * (float)n + rightArea[b + 1] * (float)rc[b + 1];
      if (cost < bestCost) { bestCost = cost; bestAxis = axis; bestSplit = b; }
    }
  }
  uint32_t mid;
  if (bestAxis < 0)
  {
    mid = first + count / 2; /* all centroids coincide: split the list in half */
  }
  else
  {
    const float ext = cbox.hi[bestAxis] - cbox.lo[bestAxis];
    const float scale = (float)ORC_BINS / ext;
    uint32_t i = first, j = first + count;
    while (i < j)
    {
      const aabb* p = &c->pb[t->prims[i]];
      int b = (int)((0.5f * (p->lo[bestAxis] + p->hi[bestAxis]) - cbox.lo[bestAxis]) * scale);
      if (b < 0) b = 0; if (b >= ORC_BINS) b = ORC_BINS - 1;
      if (b <= bestSplit) ++i; else { --j; const uint32_t tmp = t->prims[i]; t->prims[i] = t->prims[j]; t->prims[j] = tmp; }
    }
    mid = i;
    if (mid == first || mid == first + count) mid = first + count / 2;
  }
  const uint32_t left = t->numNodes; t->numNodes += 2;
  t->nodes[nodeIdx].left = left; t->nodes[nodeIdx].count = 0;
  build_rec(c, left, first, mid - first);
  build_rec(c, left + 1, mid, first + count - mid);
}

/* Inactive inputs (DESIGN.md section 3), with the bound B = 2^126 of the product's quantised boxes: a triangle with a vertex
 * coordinate that is NaN, infinite or beyond B is never hit and bounds nothing (the oracle's BVH gives it an empty box and both
 * traversal modes skip it); so is an instance whose transform has an entry that is not finite, or whose geometry's in-range
 * vertices, transformed, reach beyond B. */
static int in_range(float x) { return fabsf(x) <= 0x1p126f; }

static int tri_active(const geometry* g, uint32_t t)
{
  for (int c = 0; c < 3; ++c)
  {
    const rt_float3 v = g->attrs[g->indices[3 * t + c]].vertex;
    if (!in_range(v.x) || !in_range(v.y) || !in_range(v.z)) return 0;
  }
  return 1;
}

static void bvh_build(bvh* t, const aabb* primBoxes, uint32_t n)
{
  bvh_free(t);
  if (n == 0) return;
  t->nodes = (bnode*)malloc(sizeof(bnode) * (size_t)(2 * n));
  t->prims = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)n);
  for (uint32_t i = 0; i < n; ++i) t->prims[i] = i;
  t->numNodes = 1;
  build_ctx c = { t, primBoxes, 2 * n };
  build_rec(&c, 0, 0, n);
}

static inline float f_down(float x) { return nextafterf(x, -INFINITY); }
static inline float f_up(float x) { return nextafterf(x, INFINITY); }

void orc_scene_commit(orc_scene* s)
{
  for (int gi = 0; gi < s->numGeoms; ++gi)
  {
    geometry* g = &s->geoms[gi];
    aabb* pb = (aabb*)malloc(sizeof(aabb) * (size_t)(g->numTris ? g->numTris : 1));
    box_empty(&g->bounds);
    for (uint32_t t = 0; t < g->numTris; ++t)
    {
      box_empty(&pb[t]);
      if (!tri_active(g, t)) { for (int a = 0; a < 3; ++a) { pb[t].lo[a] = FLT_MAX; pb[t].hi[a] = -FLT_MAX; } continue; }
      for (int k = 0; k < 3; ++k)
      {
        const rt_float3 v = g->attrs[g->indices[3 * t + k]].vertex;
        const float p[3] = { v.x, v.y, v.z };
        for (int a = 0; a < 3; ++a) { if (p[a] < pb[t].lo[a]) pb[t].lo[a] = p[a]; if (p[a] > pb[t].hi[a]) pb[t].hi[a] = p[a]; }
      }
      box_grow(&g->bounds, &pb[t]);
    }
    bvh_build(&g->tree, pb, g->numTris);
    free(pb);
  }
  aabb* ib = (aabb*)malloc(sizeof(aabb) * (size_t)(s->numInsts ? s->numInsts : 1));
  for (int ii = 0; ii < s->numInsts; ++ii)
  {
    instance* in = &s->insts[ii];
    invert_3x4(in->m, in->inv);
    const aabb* gb = &s->geoms[in->geometry].bounds;
    box_empty(&in->world);
    for (int corner = 0; corner < 8; ++corner)
    {
      const double x = (corner & 1) ? gb->hi[0] : gb->lo[0];
      const double y = (corner & 2) ? gb->hi[1] : gb->lo[1];
      const double z = (corner & 4) ? gb->hi[2] : gb->lo[2];
      for (int r = 0; r < 3; ++r)
      {
        const double w = in->m[4 * r + 0] * x + in->m[4 * r + 1] * y + in->m[4 * r + 2] * z + in->m[4 * r + 3];
        /* pad: the object-space ray is a rounded transform of the world ray, so world-space bounds carry a relative slack */
        const double pad = (fabs(w) + fabs((double)gb->hi[0] - gb->lo[0]) + fabs((double)gb->hi[1] - gb->lo[1]) + fabs((double)gb->hi[2] - gb->lo[2])) * 1.0e-5;
        const float lo = f_down((float)(w - pad)), hi = f_up((float)(w + pad));
        if (lo < in->world.lo[r]) in->world.lo[r] = lo;
        if (hi > in->world.hi[r]) in->world.hi[r] = hi;
      }
    }
    if (s->geoms[in->geometry].numTris == 0 || !(gb->lo[0] <= gb->hi[0]))
      for (int k = 0; k < 3; ++k) { in->world.lo[k] = 0.0f; in->world.hi[k] = 0.0f; }
    in->active = 1;
    for (int k = 0; k < 12; ++k) in->active &= in_range(in->m[k]);
    if (in->active && s->geoms[in->geometry].numTris && gb->lo[0] <= gb->hi[0])
    {
      /* the exact world bounds of the geometry's in-range vertices (one fmaf chain per row) must lie within B */
      const geometry* g = &s->geoms[in->geometry];
      for (uint32_t v = 0; v < g->numVerts; ++v)
      {
        const float p[3] = { g->attrs[v].vertex.x, g->attrs[v].vertex.y, g->attrs[v].vertex.z };
        if (!in_range(p[0]) || !in_range(p[1]) || !in_range(p[2])) continue;
        for (int r = 0; r < 3; ++r)
          in->active &= in_range(fmaf(in->m[4 * r], p[0], fmaf(in->m[4 * r + 1], p[1], fmaf(in->m[4 * r + 2], p[2], in->m[4 * r + 3]))));
      }
    }
    if (!in->active) for (int k = 0; k < 3; ++k) { in->world.lo[k] = 0.0f; in->world.hi[k] = 0.0f; }
    else for (int k = 0; k < 3; ++k)            /* overflowing pads of the oracle's own (looser) box: keep its BVH finite */
    {
      if (!isfinite(in->world.lo[k])) in->world.lo[k] = -FLT_MAX;
      if (!isfinite(in->world.hi[k])) in->world.hi[k] = FLT_MAX;
    }
    ib[ii] = in->world;
  }
  bvh_build(&s->top, ib, (uint32_t)s->numInsts);
  free(ib);
  s->committed = 1;
}

void orc_scene_get_inverse(const orc_scene* s, int inst, float out[12]) { memcpy(out, s->insts[inst].inv, sizeof(float) * 12); }

/* ------------------------------------------------------------------------------------------
 * The ray/triangle test (DEFINED here; the reference has none -- optixTrace, raygeneration.cu:84).
 * Watertight test after Woop, Benthin, Wald, "Watertight Ray/Triangle Intersection", JCGT 2013:
 *   - per ray: kz = dominant axis of the direction, (kx, ky) the other two, swapped when dir[kz] < 0;
 *     shear Sx = d[kx]/d[kz], Sy = d[ky]/d[kz], Sz = 1/d[kz]                       (IEEE divisions)
 *   - per triangle: A,B,C = v - org; Ax = fmaf(-Sx, A[kz], A[kx]) (same for y, B, C);
 *     U = Cx*By - Cy*Bx, V = Ax*Cy - Ay*Cx, W = Bx*Ay - By*Ax with ROUNDED products (no fma, so the
 *     edge function of a shared edge is exactly antisymmetric); if any is 0, recompute all three in double;
 *     miss if signs are mixed; det = (U+V)+W, miss if 0;
 *     T = fmaf(U, Sz*A[kz], fmaf(V, Sz*B[kz], W * (Sz*C[kz]))); t = T / det      (IEEE division)
 *   - valid when tmin < t < tmax (strict), no face culling (Device.cpp:1378 flags NONE);
 *     barycentrics beta = V/det (weight of v1), gamma = W/det (weight of v2)
 *     (optixGetTriangleBarycentrics use at closesthit.cu:142-147)
 *   - closest hit = smallest t, ties broken towards the smaller (instance, primitive) pair, so the
 *     result does not depend on traversal order.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  float o[3], d[3];
  int   kx, ky, kz;
  float Sx, Sy, Sz;
  float idir[3];     /* for the slab test only (never enters a reported number) */
} oray;

static inline void oray_setup(oray* r)
{
  const float ax = fabsf(r->d[0]), ay = fabsf(r->d[1]), az = fabsf(r->d[2]);
  int kz = (ax >= ay && ax >= az) ? 0 : ((ay >= az) ? 1 : 2);
  int kx = (kz + 1) % 3, ky = (kx + 1) % 3;
  if (r->d[kz] < 0.0f) { const int t = kx; kx = ky; ky = t; }
  r->kx = kx; r->ky = ky; r->kz = kz;
  r->Sx = r->d[kx] / r->d[kz];
  r->Sy = r->d[ky] / r->d[kz];
  r->Sz = 1.0f / r->d[kz];
  for (int k = 0; k < 3; ++k)
  {
    float d = r->d[k];
    if (fabsf(d) < 0x1p-80f) d = copysignf(0x1p-80f, d);
    r->idir[k] = 1.0f / d;
  }
}

/* returns 1 and fills t,beta,gamma when the line through the ray pierces the triangle at a finite t */
static inline int tri_test(const oray* r, const float* v0, const float* v1, const float* v2, float* t, float* beta, float* gamma)
{
  const int kx = r->kx, ky = r->ky, kz = r->kz;
  const float A[3] = { v0[0] - r->o[0], v0[1] - r->o[1], v0[2] - r->o[2] };
  const float B[3] = { v1[0] - r->o[0], v1[1] - r->o[1], v1[2] - r->o[2] };
  const float C[3] = { v2[0] - r->o[0], v2[1] - r->o[1], v2[2] - r->o[2] };
  const float Ax = fmaf(-r->Sx, A[kz], A[kx]), Ay = fmaf(-r->Sy, A[kz], A[ky]);
  const float Bx = fmaf(-r->Sx, B[kz], B[kx]), By = fmaf(-r->Sy, B[kz], B[ky]);
  const float Cx = fmaf(-r->Sx, C[kz], C[kx]), Cy = fmaf(-r->Sy, C[kz], C[ky]);
  float U = Cx * By - Cy * Bx;
  float V = Ax * Cy - Ay * Cx;
  float W = Bx * Ay - By * Ax;
  if (U == 0.0f || V == 0.0f || W == 0.0f)
  {
    U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
    V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
    W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
  }
  if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return 0;
  const float det = (U + V) + W;
  if (det == 0.0f) return 0;
  const float Az = r->Sz * A[kz], Bz = r->Sz * B[kz], Cz = r->Sz * C[kz];
  const float T = fmaf(U, Az, fmaf(V, Bz, W * Cz));
  *t = T / det;
  *beta = V / det;
  *gamma = W / det;
  return 1;
}

/* slab test against a box, padded so that it can never cull a triangle hit the test above reports */
static inline int box_test(const oray* r, const aabb* b, float tmin, float tmax)
{
  float tn = tmin, tf = tmax;
  for (int k = 0; k < 3; ++k)
  {
    const float t0 = (b->lo[k] - r->o[k]) * r->idir[k];
    const float t1 = (b->hi[k] - r->o[k]) * r->idir[k];
    float lo = t0 < t1 ? t0 : t1, hi = t0 < t1 ? t1 : t0;
    lo -= fabsf(lo) * 0x1p-18f; hi += fabsf(hi) * 0x1p-18f;
    if (lo > tn) tn = lo;
    if (hi < tf) tf = hi;
  }
  return tn <= tf;
}

/* skip != NULL: only candidates that come AFTER the skip key in the canonical order (t, instance, primitive) count */
typedef struct { float t; uint32_t inst, prim; } hitkey;
typedef struct { float t, u, v; uint32_t inst, prim; const hitkey* skip; } besthit;

static inline void consider(besthit* best, float t, float u, float v, uint32_t inst, uint32_t prim, float tmin, float tmax)
{
  if (!(t > tmin && t < tmax)) return;
  if (best->skip)
  {
    const hitkey* k = best->skip;
    if (!(t > k->t || (t == k->t && (inst > k->inst || (inst == k->inst && prim > k->prim))))) return;
  }
  if (best->inst != 0xffffffffu)
  {
    if (t > best->t) return;
    if (t == best->t && (inst > best->inst || (inst == best->inst && prim >= best->prim))) return;
  }
  best->t = t; best->u = u; best->v = v; best->inst = inst; best->prim = prim;
}

static inline void tri_verts(const geometry* g, uint32_t prim, const float** v0, const float** v1, const float** v2)
{
  const uint32_t* ix = &g->indices[3u * prim];
  *v0 = &g->attrs[ix[0]].vertex.x; *v1 = &g->attrs[ix[1]].vertex.x; *v2 = &g->attrs[ix[2]].vertex.x;
}

/* world ray -> object ray of one instance: fmaf chains, direction NOT normalised so t is shared */
static inline void to_object(const float inv[12], const float o[3], const float d[3], oray* r)
{
  for (int k = 0; k < 3; ++k)
  {
    const float* m = &inv[4 * k];
    r->o[k] = fmaf(m[0], o[0], fmaf(m[1], o[1], fmaf(m[2], o[2], m[3])));
    r->d[k] = fmaf(m[0], d[0], fmaf(m[1], d[1], m[2] * d[2]));
  }
  oray_setup(r);
}

/* anyHit != 0: return at the first valid hit.  Returns 1 if a hit was found. */
static int trace_instance(const orc_scene* s, uint32_t ii, const float o[3], const float d[3], float tmin, float tmax,
                          int mode, int anyHit, besthit* best, orc_stats* st)
{
  const instance* in = &s->insts[ii];
  const geometry* g = &s->geoms[in->geometry];
  if (g->numTris == 0 || !in->active) return 0;
  oray r; to_object(in->inv, o, d, &r);
  if (st) st->instancesEntered++;
  const float *v0, *v1, *v2; float t, u, v;
  if (mode == 1)
  {
    for (uint32_t p = 0; p < g->numTris; ++p)
    {
      if (!tri_active(g, p)) continue;
      tri_verts(g, p, &v0, &v1, &v2);
      if (st) st->trisTested++;
      if (tri_test(&r, v0, v1, v2, &t, &u, &v))
      {
        if (anyHit) { if (t > tmin && t < tmax) return 1; }
        else consider(best, t, u, v, ii, p, tmin, tmax);
      }
    }
    return 0;
  }
  uint32_t stack[64]; int sp = 0; stack[sp++] = 0;
  while (sp)
  {
    const bnode* n = &g->tree.nodes[stack[--sp]];
    const float far = (!anyHit && best->inst != 0xffffffffu) ? best->t : tmax;
    if (st) st->nodesVisited++;
    if (!box_test(&r, &n->box, tmin, far)) continue;
    if (n->count)
    {
      for (uint32_t i = n->left; i < n->left + n->count; ++i)
      {
        const uint32_t p = g->tree.prims[i];
        if (!tri_active(g, p)) continue;
        tri_verts(g, p, &v0, &v1, &v2);
        if (st) st->trisTested++;
        if (tri_test(&r, v0, v1, v2, &t, &u, &v))
        {
          if (anyHit) { if (t > tmin && t < tmax) return 1; }
          else consider(best, t, u, v, ii, p, tmin, tmax);
        }
      }
    }
    else if (sp + 2 <= 64)
    {
      /* nearer child (by box centre along the dominant axis) on top */
      const bnode* l = &g->tree.nodes[n->left];
      const bnode* rr = &g->tree.nodes[n->left + 1];
      const int k = r.kz;
      const float cl = (l->box.lo[k] + l->box.hi[k]) * r.d[k], cr = (rr->box.lo[k] + rr->box.hi[k]) * r.d[k];
      if (cl < cr) { stack[sp++] = n->left + 1; stack[sp++] = n->left; }
      else         { stack[sp++] = n->left; stack[sp++] = n->left + 1; }
    }
  }
  return 0;
}

static int trace_scene_after(const orc_scene* s, const float o[3], const float d[3], float tmin, float tmax,
                             int mode, int anyHit, besthit* best, orc_stats* st, const hitkey* skip)
{
  best->inst = 0xffffffffu; best->prim = 0xffffffffu; best->t = -1.0f; best->u = 0.0f; best->v = 0.0f; best->skip = skip;
  if (!(tmax > tmin)) return 0;
  if (mode == 1 || s->top.numNodes == 0)
  {
    for (int ii = 0; ii < s->numInsts; ++ii)
      if (trace_instance(s, (uint32_t)ii, o, d, tmin, tmax, mode, anyHit, best, st)) return 1;
    return (!anyHit && best->inst != 0xffffffffu);
  }
  oray w; memcpy(w.o, o, sizeof(w.o)); memcpy(w.d, d, sizeof(w.d)); oray_setup(&w);
  uint32_t stack[64]; int sp = 0; stack[sp++] = 0;
  while (sp)
  {
    const bnode* n = &s->top.nodes[stack[--sp]];
    const float far = (!anyHit && best->inst != 0xffffffffu) ? best->t : tmax;
    if (st) st->nodesVisited++;
    if (!box_test(&w, &n->box, tmin, far)) continue;
    if (n->count)
    {
      for (uint32_t i = n->left; i < n->left + n->count; ++i)
        if (trace_instance(s, s->top.prims[i], o, d, tmin, tmax, mode, anyHit, best, st)) return 1;
    }
    else if (sp + 2 <= 64)
    {
      stack[sp++] = n->left; stack[sp++] = n->left + 1;
    }
  }
  return (!anyHit && best->inst != 0xffffffffu);
}

static int trace_scene(const orc_scene* s, const float o[3], const float d[3], float tmin, float tmax,
                       int mode, int anyHit, besthit* best, orc_stats* st)
{
  return trace_scene_after(s, o, d, tmin, tmax, mode, anyHit, best, st, NULL);
}

/* Closest hit that comes after (skipT, skipInst, skipPrim) in the canonical candidate order; the building block of the
 * ordered any-hit processing below (exported for the reference driver, which runs the reference's own any-hit programs). */
void orc_trace_closest_after(const orc_scene* s, const orc_ray* ray, float skipT, uint32_t skipInst, uint32_t skipPrim, orc_hit* hit)
{
  const float o[3] = { ray->ox, ray->oy, ray->oz }, d[3] = { ray->dx, ray->dy, ray->dz };
  const hitkey k = { skipT, skipInst, skipPrim };
  besthit b;
  trace_scene_after(s, o, d, ray->tmin, ray->tmax, 0, 0, &b, NULL, &k);
  hit->t = b.t; hit->u = b.u; hit->v = b.v; hit->inst = b.inst; hit->prim = b.prim;
}

void orc_trace_closest(const orc_scene* s, const orc_ray* rays, uint64_t n, int mode, orc_hit* hits, orc_stats* stats)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    const float o[3] = { rays[i].ox, rays[i].oy, rays[i].oz }, d[3] = { rays[i].dx, rays[i].dy, rays[i].dz };
    besthit b;
    trace_scene(s, o, d, rays[i].tmin, rays[i].tmax, mode, 0, &b, stats);
    hits[i].t = b.t; hits[i].u = b.u; hits[i].v = b.v; hits[i].inst = b.inst; hits[i].prim = b.prim;
    if (stats) stats->radianceRays++;
  }
}

void orc_trace_any(const orc_scene* s, const orc_ray* rays, uint64_t n, int mode, uint8_t* occluded, orc_stats* stats)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    const float o[3] = { rays[i].ox, rays[i].oy, rays[i].oz }, d[3] = { rays[i].dx, rays[i].dy, rays[i].dz };
    besthit b;
    occluded[i] = (uint8_t)trace_scene(s, o, d, rays[i].tmin, rays[i].tmax, mode, 1, &b, stats);
    if (stats) stats->shadowRays++;
  }
}

/* ------------------------------------------------------------------------------------------
 * Environment texture lookup (DEFINED: software bilinear filter, wrap in u, clamp in v, texel
 * centres at (i+0.5)/W; replaces tex2D at miss.cu:90 and light_sample.cu:147).
 * ------------------------------------------------------------------------------------------ */
static v3 env_lookup(const orc_scene* s, float u, float v)
{
  const int W = (int)s->envW, H = (int)s->envH;
  const float x = u * (float)W - 0.5f, y = v * (float)H - 0.5f;
  const float fx = floorf(x), fy = floorf(y);
  const float ax = x - fx, ay = y - fy;
  int x0 = (int)fx % W; if (x0 < 0) x0 += W;
  int x1 = x0 + 1; if (x1 >= W) x1 = 0;
  int y0 = (int)fy, y1 = y0 + 1;
  if (y0 < 0) y0 = 0; if (y0 > H - 1) y0 = H - 1;
  if (y1 < 0) y1 = 0; if (y1 > H - 1) y1 = H - 1;
  const float* t00 = &s->envTexels[4 * ((size_t)y0 * W + x0)];
  const float* t10 = &s->envTexels[4 * ((size_t)y0 * W + x1)];
  const float* t01 = &s->envTexels[4 * ((size_t)y1 * W + x0)];
  const float* t11 = &s->envTexels[4 * ((size_t)y1 * W + x1)];
  float c[3];
  for (int k = 0; k < 3; ++k)
  {
    const float a = t00[k] + ax * (t10[k] - t00[k]);
    const float b = t01[k] + ax * (t11[k] - t01[k]);
    c[k] = a + ay * (b - a);
  }
  return V3(c[0], c[1], c[2]);
}

/* ------------------------------------------------------------------------------------------
 * Material textures (MaterialDefinition.textureAlbedo / textureCutout; tex2D at closesthit.cu:235, anyhit.cu:70, :119).
 * The reference samples CUDA texture objects created with wrap/wrap addressing, linear filtering and normalised
 * coordinates (src/Texture.cpp:670-675).  DEFINED here like the environment lookup: a handle is the address of a
 * 16-byte header {uint32 width, height, 0, 0} followed by width*height RGBA32F texels; software bilinear filter,
 * wrap in u AND v, texel centres at (i+0.5)/W.
 * ------------------------------------------------------------------------------------------ */
static v3 tex2d_wrap(uint64_t handle, float u, float v)
{
  const uint32_t* header = (const uint32_t*)(uintptr_t)handle;
  const float* texels = (const float*)(header + 4);
  const int W = (int)header[0], H = (int)header[1];
  const float x = u * (float)W - 0.5f, y = v * (float)H - 0.5f;
  const float fx = floorf(x), fy = floorf(y);
  const float ax = x - fx, ay = y - fy;
  int x0 = (int)fx % W; if (x0 < 0) x0 += W;
  int x1 = x0 + 1; if (x1 >= W) x1 = 0;
  int y0 = (int)fy % H; if (y0 < 0) y0 += H;
  int y1 = y0 + 1; if (y1 >= H) y1 = 0;
  const float* t00 = &texels[4 * ((size_t)y0 * W + x0)];
  const float* t10 = &texels[4 * ((size_t)y0 * W + x1)];
  const float* t01 = &texels[4 * ((size_t)y1 * W + x0)];
  const float* t11 = &texels[4 * ((size_t)y1 * W + x1)];
  float c[3];
  for (int k = 0; k < 3; ++k)
  {
    const float a = t00[k] + ax * (t10[k] - t00[k]);
    const float b = t01[k] + ax * (t11[k] - t01[k]);
    c[k] = a + ay * (b - a);
  }
  return V3(c[0], c[1], c[2]);
}

void orc_tex2d(uint64_t handle, float u, float v, float out[3])
{
  const v3 c = tex2d_wrap(handle, u, v);
  out[0] = c.x; out[1] = c.y; out[2] = c.z;
}

/* ------------------------------------------------------------------------------------------
 * Per-ray data, surface state (shaders/per_ray_data.h:84-114, shader_common.h State)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  v3 pos; float distance;
  v3 wo, wi;
  v3 radiance; uint32_t flags;
  v3 f_over_pdf; float pdf;
  v3 sigma_t; v2 ior;
  v4 absorption_ior;
  uint32_t seed;
} prd_t;

typedef struct { v3 normalGeo, tangent, normal, texcoord, albedo; } state_t;

typedef struct { v3 tangent, bitangent, normal; } tbn_t;

/* shader_common.h:118-124 */
static inline tbn_t tbn_make(v3 tangent_reference, v3 n)
{
  tbn_t t;
  t.normal = n;
  t.bitangent = vnormalize(vcross(n, tangent_reference));
  t.tangent = vcross(t.bitangent, n);
  return t;
}
static inline v3 tbn_to_local(const tbn_t* t, v3 p) { return V3(vdot(p, t->tangent), vdot(p, t->bitangent), vdot(p, t->normal)); }
static inline v3 tbn_to_world(const tbn_t* t, v3 p)
{
  return vadd(vadd(vscale(t->tangent, p.x), vscale(t->bitangent, p.y)), vscale(t->normal, p.z));
}

/* shader_common.h:47-78 */
static int refract_dir(v3* r, v3 i, v3 n, float ior)
{
  v3 nn = n;
  float negNdotV = vdot(i, nn);
  float eta;
  if (negNdotV > 0.0f) { eta = ior; nn = vneg(n); negNdotV = -negNdotV; }
  else                 { eta = 1.f / ior; }
  const float k = 1.f - eta * eta * (1.f - negNdotV * negNdotV);
  if (k < 0.0f) { *r = v3s(0.f); return 0; }
  *r = vnormalize(vsub(vscale(i, eta), vscale(nn, eta * negNdotV + sqrtf(k))));
  return 1;
}

/* bxdf_specular.cu:42-69 (duplicated at bxdf_ggx_smith.cu:45-72) */
static float fresnel_dielectric(float et, float cosIn)
{
  const float cosi = fabsf(cosIn);
  float sint = 1.0f - cosi * cosi;
  sint = (0.0f < sint) ? sqrtf(sint) / et : 0.0f;
  if (1.0f < sint) return 1.0f;
  float cost = 1.0f - sint * sint;
  cost = (0.0f < cost) ? sqrtf(cost) : 0.0f;
  const float et_cosi = et * cosi, et_cost = et * cost;
  const float rPerp = (cosi - et_cost) / (cosi + et_cost);
  const float rPar  = (et_cosi - cost) / (et_cosi + cost);
  const float result = (rPar * rPar + rPerp * rPerp) * 0.5f;
  return (result <= 1.0f) ? result : 1.0f;
}

/* ---- brdf_diffuse (bxdf_diffuse.cu:39-95) ---- */
static void align_vector(v3 axis, v3* w)
{
  const float s = copysignf(1.0f, axis.z);
  w->z *= s;
  const v3 h = V3(axis.x, axis.y, axis.z + s);
  const float k = vdot(*w, h) / (1.0f + fabsf(axis.z));
  *w = vsub(vscale(h, k), *w);
}

static void sample_brdf_diffuse(const rt_MaterialDefinition* m, const state_t* st, prd_t* prd)
{
  (void)m;
  const v2 sample = rng2(&prd->seed);
  const float theta = 2.0f * RT_PI_F * sample.x;
  const float r = sqrtf(sample.y);
  v3 w;
  w.x = r * rt_cosf(theta);
  w.y = r * rt_sinf(theta);
  w.z = 1.0f - w.x * w.x - w.y * w.y;
  w.z = (0.0f < w.z) ? sqrtf(w.z) : 0.0f;
  prd->pdf = w.z * RT_1_PI_F;
  align_vector(st->normal, &w);
  prd->wi = w;
  if (prd->pdf <= 0.0f || vdot(prd->wi, st->normalGeo) <= 0.0f) { prd->flags |= RT_FLAG_TERMINATE; return; }
  prd->f_over_pdf = st->albedo;
  prd->flags |= RT_FLAG_DIFFUSE;
}

static v4 eval_brdf_diffuse(const rt_MaterialDefinition* m, const state_t* st, const prd_t* prd, v3 wiL)
{
  (void)m; (void)prd;
  const v3 f = vscale(st->albedo, RT_1_PI_F);
  const float pdf = fmaxf(0.0f, vdot(wiL, st->normal) * RT_1_PI_F);
  v4 r = { f.x, f.y, f.z, pdf };
  return r;
}

/* ---- brdf_specular / bsdf_specular (bxdf_specular.cu:71-134) ---- */
static void sample_brdf_specular(const rt_MaterialDefinition* m, const state_t* st, prd_t* prd)
{
  (void)m;
  prd->wi = vreflect(vneg(prd->wo), st->normal);
  if (vdot(prd->wi, st->normalGeo) <= 0.0f) { prd->flags |= RT_FLAG_TERMINATE; return; }
  prd->f_over_pdf = st->albedo;
  prd->pdf = 1.0f;
}

static void sample_bsdf_specular(const rt_MaterialDefinition* m, const state_t* st, prd_t* prd)
{
  prd->absorption_ior.x = m->absorption.x; prd->absorption_ior.y = m->absorption.y;
  prd->absorption_ior.z = m->absorption.z; prd->absorption_ior.w = m->ior;
  const float eta = (prd->flags & (RT_FLAG_FRONTFACE | RT_FLAG_THINWALLED))
                  ? prd->absorption_ior.w / prd->ior.x
                  : prd->ior.y / prd->absorption_ior.w;
  const v3 R = vreflect(vneg(prd->wo), st->normal);
  float reflective = 1.0f;
  if (refract_dir(&prd->wi, vneg(prd->wo), st->normal, eta))
  {
    if (prd->flags & RT_FLAG_THINWALLED) prd->wi = vneg(prd->wo);
    reflective = fresnel_dielectric(eta, vdot(prd->wo, st->normal));
  }
  const float pseudo = orc_rng(&prd->seed);
  if (pseudo < reflective) prd->wi = R;
  else if (!(prd->flags & RT_FLAG_THINWALLED)) prd->flags |= RT_FLAG_TRANSMISSION;
  prd->f_over_pdf = st->albedo;
  prd->pdf = 1.0f;
}

/* ---- GGX-Smith (bxdf_ggx_smith.cu:74-319) ---- */
static v2 ggx_d_pdf(float ax, float ay, v3 wm)
{
  v2 r = { 0.0f, 0.0f };
  if (RT_DENOMINATOR_EPSILON < wm.z)
  {
    const float cosThetaSqr = wm.z * wm.z;
    const float tanThetaSqr = (1.0f - cosThetaSqr) / cosThetaSqr;
    const float phiM = rt_atan2f(wm.y, wm.x);
    const float cosPhiM = rt_cosf(phiM), sinPhiM = rt_sinf(phiM);
    const float term = 1.0f + tanThetaSqr * ((cosPhiM * cosPhiM) / (ax * ax) + (sinPhiM * sinPhiM) / (ay * ay));
    const float d = 1.0f / (RT_PI_F * ax * ay * cosThetaSqr * cosThetaSqr * term * term);
    r.x = d; r.y = d * wm.z;
  }
  return r;
}

static v3 ggx_sample(float ax, float ay, float u1, float u2)
{
  const float theta = rt_atanf(ay * sqrtf(u1) / sqrtf(1.0f - u1));
  const float phi = 2.0f * RT_PI_F * u2;
  const float sinTheta = rt_sinf(theta);
  return vnormalize(V3(rt_cosf(phi) * sinTheta * ax / ay, rt_sinf(phi) * sinTheta, rt_cosf(theta)));
}

static float smith_g1(float alpha, v3 w, v3 wm)
{
  const float w_wm = vdot(w, wm);
  if (w_wm * w.z <= 0.0f) return 0.0f;
  const float cosThetaSqr = w.z * w.z;
  const float sinThetaSqr = 1.0f - cosThetaSqr;
  const float tanThetaSqr = (0.0f < sinThetaSqr) ? sinThetaSqr / cosThetaSqr : 0.0f;
  const float invASqr = alpha * alpha * tanThetaSqr;
  return 2.0f / (1.0f + sqrtf(1.0f + invASqr));
}

static float ggx_g(float ax, float ay, v3 wo, v3 wi, v3 wm)
{
  float phi = rt_atan2f(wo.y, wo.x);
  float c = rt_cosf(phi), sn = rt_sinf(phi);
  float alpha = sqrtf(c * c * ax * ax + sn * sn * ay * ay);
  const float g = smith_g1(alpha, wo, wm);
  phi = rt_atan2f(wi.y, wi.x);
  c = rt_cosf(phi); sn = rt_sinf(phi);
  alpha = sqrtf(c * c * ax * ax + sn * sn * ay * ay);
  return g * smith_g1(alpha, wi, wm);
}

static void sample_brdf_ggx(const rt_MaterialDefinition* m, const state_t* st, prd_t* prd)
{
  const v2 sample = rng2(&prd->seed);
  const v3 wm = ggx_sample(m->roughness.x, m->roughness.y, sample.x, sample.y);
  const tbn_t ts = tbn_make(st->tangent, st->normal);
  const v3 wh = tbn_to_world(&ts, wm);
  prd->wi = vreflect(vneg(prd->wo), wh);
  if (vdot(prd->wi, st->normalGeo) <= 0.0f) { prd->flags |= RT_FLAG_TERMINATE; return; }
  const v3 wo = tbn_to_local(&ts, prd->wo);
  const v3 wi = tbn_to_local(&ts, prd->wi);
  const float wi_wh = vdot(prd->wi, wh);
  if (wo.z <= 0.0f || wi.z <= 0.0f || wi_wh <= 0.0f) { prd->flags |= RT_FLAG_TERMINATE; return; }
  const v2 D_PDF = ggx_d_pdf(m->roughness.x, m->roughness.y, wm);
  if (D_PDF.y <= 0.0f) { prd->flags |= RT_FLAG_TERMINATE; return; }
  const float G = ggx_g(m->roughness.x, m->roughness.y, wo, wi, wm);
  prd->pdf = D_PDF.y / (4.0f * wi_wh);
  prd->f_over_pdf = vscale(st->albedo, G * D_PDF.x * wi_wh / (D_PDF.y * wo.z));
  prd->flags |= RT_FLAG_DIFFUSE;
}

static v4 eval_brdf_ggx(const rt_MaterialDefinition* m, const state_t* st, const prd_t* prd, v3 wiL)
{
  const v4 zero = { 0.0f, 0.0f, 0.0f, 0.0f };
  const tbn_t ts = tbn_make(st->tangent, st->normal);
  const v3 wo = tbn_to_local(&ts, prd->wo);
  const v3 wi = tbn_to_local(&ts, wiL);
  if (wo.z <= 0.0f || wi.z <= 0.0f) return zero;
  v3 wm = vadd(wo, wi);
  if (v3_is_null(wm)) return zero;
  wm = vnormalize(wm);
  const v2 D_PDF = ggx_d_pdf(m->roughness.x, m->roughness.y, wm);
  const float G = ggx_g(m->roughness.x, m->roughness.y, wo, wi, wm);
  const v3 f = vscale(st->albedo, D_PDF.x * G / (4.0f * wo.z * wi.z));
  const float pdf = D_PDF.y / (4.0f * vdot(wi, wm));
  v4 r = { f.x, f.y, f.z, pdf };
  return r;
}

static void sample_bsdf_ggx(const rt_MaterialDefinition* m, const state_t* st, prd_t* prd)
{
  prd->absorption_ior.x = m->absorption.x; prd->absorption_ior.y = m->absorption.y;
  prd->absorption_ior.z = m->absorption.z; prd->absorption_ior.w = m->ior;
  const float eta = (prd->flags & (RT_FLAG_FRONTFACE | RT_FLAG_THINWALLED))
                  ? prd->absorption_ior.w / prd->ior.x
                  : prd->ior.y / prd->absorption_ior.w;
  const v2 sample = rng2(&prd->seed);
  const v3 wm = ggx_sample(m->roughness.x, m->roughness.y, sample.x, sample.y);
  const tbn_t ts = tbn_make(st->tangent, st->normal);
  const v3 wh = tbn_to_world(&ts, wm);
  const v3 R = vreflect(vneg(prd->wo), wh);
  float reflective = 1.0f;
  if (refract_dir(&prd->wi, vneg(prd->wo), wh, eta))
  {
    if (prd->flags & RT_FLAG_THINWALLED) prd->wi = vreflect(R, st->normal);
    reflective = fresnel_dielectric(eta, vdot(prd->wo, wh));
  }
  const float pseudo = orc_rng(&prd->seed);
  if (pseudo < reflective) prd->wi = R;
  else if (!(prd->flags & RT_FLAG_THINWALLED)) prd->flags |= RT_FLAG_TRANSMISSION;
  prd->f_over_pdf = st->albedo;
  prd->pdf = 1.0f;
}

/* callable table: closesthit.cu:246-248 (sample = 3+2+indexBSDF*2, eval = +1); eval of every specular
 * lobe is eval_brdf_specular = 0 (Device.cpp:744-748, 768-772). */
static void bsdf_sample(const rt_MaterialDefinition* m, const state_t* st, prd_t* prd)
{
  switch (m->indexBSDF)
  {
    default:
    case RT_BRDF_DIFFUSE:   sample_brdf_diffuse(m, st, prd); break;
    case RT_BRDF_SPECULAR:  sample_brdf_specular(m, st, prd); break;
    case RT_BSDF_SPECULAR:  sample_bsdf_specular(m, st, prd); break;
    case RT_BRDF_GGX_SMITH: sample_brdf_ggx(m, st, prd); break;
    case RT_BSDF_GGX_SMITH: sample_bsdf_ggx(m, st, prd); break;
  }
}

static v4 bsdf_eval(const rt_MaterialDefinition* m, const state_t* st, const prd_t* prd, v3 wiL)
{
  const v4 zero = { 0.0f, 0.0f, 0.0f, 0.0f };
  switch (m->indexBSDF)
  {
    case RT_BRDF_DIFFUSE:   return eval_brdf_diffuse(m, st, prd, wiL);
    case RT_BRDF_GGX_SMITH: return eval_brdf_ggx(m, st, prd, wiL);
    default:                return zero;
  }
}

/* ---- lights (light_sample.cu:42-177) ---- */
typedef struct { v3 position; int index; v3 direction; float distance; v3 emission; float pdf; } light_sample_t;

static void light_env_constant(const orc_scene* s, int numLights, v3 point, v2 sample, light_sample_t* ls)
{
  (void)s; (void)point;
  v3 p;
  p.z = 1.0f - 2.0f * sample.x;
  float r = 1.0f - p.z * p.z;
  r = (0.0f < r) ? sqrtf(r) : 0.0f;
  const float phi = sample.y * 2.0f * RT_PI_F;
  p.x = r * rt_cosf(phi);
  p.y = r * rt_sinf(phi);
  ls->direction = p;
  ls->pdf = 0.25f * RT_1_PI_F;
  ls->distance = RT_DEFAULT_MAX;
  ls->emission = v3s((float)numLights);
}

static void light_env_sphere(const orc_scene* s, int numLights, float envRotation, v3 point, v2 sample, light_sample_t* ls)
{
  (void)point;
  const unsigned int sizeV = s->envH;
  unsigned int ilo = 0, ihi = sizeV;
  const float* cdfV = s->envCdfV;
  while (ilo != ihi - 1)
  {
    const unsigned int i = (ilo + ihi) >> 1;
    if (sample.y < cdfV[i]) ihi = i; else ilo = i;
  }
  const unsigned int vIdx = ilo;
  const unsigned int sizeU = s->envW;
  ilo = 0; ihi = sizeU;
  const float* cdfU = &s->envCdfU[(size_t)vIdx * (sizeU + 1)];
  while (ilo != ihi - 1)
  {
    const unsigned int i = (ilo + ihi) >> 1;
    if (sample.x < cdfU[i]) ihi = i; else ilo = i;
  }
  const unsigned int uIdx = ilo;
  const float cdfLowerU = cdfU[uIdx], cdfUpperU = cdfU[uIdx + 1];
  const float du = (sample.x - cdfLowerU) / (cdfUpperU - cdfLowerU);
  const float cdfLowerV = cdfV[vIdx], cdfUpperV = cdfV[vIdx + 1];
  const float dv = (sample.y - cdfLowerV) / (cdfUpperV - cdfLowerV);
  const float u = ((float)uIdx + du) / (float)sizeU;
  const float v = ((float)vIdx + dv) / (float)sizeV;
  const float phi = (u - envRotation) * 2.0f * RT_PI_F;
  const float theta = v * RT_PI_F;
  const float sinTheta = rt_sinf(theta);
  ls->direction = V3(-rt_sinf(phi) * sinTheta, -rt_cosf(theta), rt_cosf(phi) * sinTheta);
  ls->distance = RT_DEFAULT_MAX;
  const v3 emission = env_lookup(s, u, v);
  ls->emission = vscale(emission, (float)numLights);
  ls->pdf = intensity3(emission) / s->envIntegral;
}

static void light_parallelogram(const orc_scene* s, int numLights, v3 point, v2 sample, light_sample_t* ls)
{
  ls->pdf = 0.0f;
  const rt_LightDefinition* light = &s->lights[ls->index];
  ls->position = vadd(vadd(from_f3(light->position), vscale(from_f3(light->vecU), sample.x)), vscale(from_f3(light->vecV), sample.y));
  ls->direction = vsub(ls->position, point);
  ls->distance = vlength(ls->direction);
  if (RT_DENOMINATOR_EPSILON < ls->distance)
  {
    ls->direction = vdivs(ls->direction, ls->distance);
    const float cosTheta = vdot(vneg(ls->direction), from_f3(light->normal));
    if (RT_DENOMINATOR_EPSILON < cosTheta)
    {
      ls->emission = vscale(from_f3(light->emission), (float)numLights);
      ls->pdf = (ls->distance * ls->distance) / (light->area * cosTheta);
    }
  }
}

/* ---- lens shaders (lens_shader.cu:40-99) ---- */
static void lens_shader(const orc_scene* s, int lens, v2 screen, v2 pixel, v2 sample, v3* origin, v3* direction)
{
  const rt_CameraDefinition* cam = &s->camera;
  const v3 cP = from_f3(cam->P), cU = from_f3(cam->U), cV = from_f3(cam->V), cW = from_f3(cam->W);
  *origin = cP;
  if (lens == RT_LENS_FISHEYE)
  {
    const v2 fragment = { pixel.x + sample.x, pixel.y + sample.y };
    const v2 center = { screen.x * 0.5f, screen.y * 0.5f };
    const float invLen = 1.0f / sqrtf(center.x * center.x + center.y * center.y);
    const v2 uv = { (fragment.x - center.x) * invLen, (fragment.y - center.y) * invLen };
    const float z = rt_cosf(sqrtf(uv.x * uv.x + uv.y * uv.y) * 0.7071067812f * 0.5f * RT_PI_F);
    const v3 U = vnormalize(cU), V = vnormalize(cV), W = vnormalize(cW);
    *direction = vnormalize(vadd(vadd(vscale(U, uv.x), vscale(V, uv.y)), vscale(W, z)));
  }
  else if (lens == RT_LENS_SPHERE)
  {
    const v2 uv = { (pixel.x + sample.x) / screen.x, (pixel.y + sample.y) / screen.y };
    const float phi = uv.x * 2.0f * RT_PI_F;
    const float theta = uv.y * RT_PI_F;
    const float sinTheta = rt_sinf(theta);
    const v3 v = V3(-rt_sinf(phi) * sinTheta, -rt_cosf(theta), -rt_cosf(phi) * sinTheta);
    const v3 U = vnormalize(cU), V = vnormalize(cV), W = vnormalize(cW);
    *direction = vnormalize(vadd(vadd(vscale(U, v.x), vscale(V, v.y)), vscale(W, v.z)));
  }
  else
  {
    const v2 fragment = { pixel.x + sample.x, pixel.y + sample.y };
    const v2 ndc = { (fragment.x / screen.x) * 2.0f - 1.0f, (fragment.y / screen.y) * 2.0f - 1.0f };
    *direction = vnormalize(vadd(vadd(vscale(cU, ndc.x), vscale(cV, ndc.y)), cW));
  }
}

/* ---- miss programs (miss.cu:41-109) ---- */
static void miss_program(const orc_scene* s, int miss, float envRotation, prd_t* prd)
{
  if (miss == RT_MISS_CONSTANT)
  {
    const float w = (prd->flags & RT_FLAG_DIFFUSE) ? power_heuristic(prd->pdf, 0.25f * RT_1_PI_F) : 1.0f;
    prd->radiance = v3s(w);
  }
  else if (miss == RT_MISS_SPHERE)
  {
    const v3 R = prd->wi;
    const float u = (rt_atan2f(R.x, -R.z) + RT_PI_F) * 0.5f * RT_1_PI_F + envRotation;
    const float theta = rt_acosf(-R.y);
    const float v = theta * RT_1_PI_F;
    const v3 emission = env_lookup(s, u, v);
    float w = 1.0f;
    if (prd->flags & RT_FLAG_DIFFUSE)
    {
      const float pdfLight = intensity3(emission) / s->envIntegral;
      w = power_heuristic(prd->pdf, pdfLight);
    }
    prd->radiance = vscale(emission, w);
  }
  else
  {
    prd->radiance = v3s(0.0f);
  }
  prd->flags |= RT_FLAG_TERMINATE;
}

/* ---- closest hit (closesthit.cu:126-305) ---- */
static inline v3 xf_vector(const float* m, v3 v)
{
  return V3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[4] * v.x + m[5] * v.y + m[6] * v.z, m[8] * v.x + m[9] * v.y + m[10] * v.z);
}
static inline v3 xf_normal(const float* inv, v3 v)
{
  return V3(inv[0] * v.x + inv[4] * v.y + inv[8] * v.z, inv[1] * v.x + inv[5] * v.y + inv[9] * v.z, inv[2] * v.x + inv[6] * v.y + inv[10] * v.z);
}

typedef struct {
  const orc_scene* s; const rt_SystemData* sys; int miss; int mode; orc_stats* st;
} shade_ctx;

/* ------------------------------------------------------------------------------------------
 * Cutout opacity: __anyhit__radiance_cutout / __anyhit__shadow_cutout (anyhit.cu:46-80, :94-132).
 *
 * OptiX runs an any-hit program for candidate intersections in an unspecified order and each invocation may draw one
 * random number from the path's seed, so the reference's result depends on the driver's traversal order.  DEFINED
 * here: candidates are processed in the canonical order (t, instance, primitive) ascending, i.e. the closest candidate
 * first; an ignored candidate is followed by the next one in that order.  The instance's hit records are the cutout
 * ones exactly when its material has a cutout texture (src/Device.cpp:1503-1513, :1141-1160).
 * ------------------------------------------------------------------------------------------ */
static float cutout_opacity(const orc_scene* s, const rt_MaterialDefinition* material, const besthit* hit)
{
  const instance* in = &s->insts[hit->inst];
  const geometry* g = &s->geoms[in->geometry];
  const uint32_t* tri = &g->indices[3u * hit->prim];
  const float bx = hit->u, by = hit->v;
  const float alpha = 1.0f - bx - by;
  const v3 texcoord = vadd(vadd(vscale(from_f3(g->attrs[tri[0]].texcoord), alpha), vscale(from_f3(g->attrs[tri[1]].texcoord), bx)),
                           vscale(from_f3(g->attrs[tri[2]].texcoord), by));
  return intensity3(tex2d_wrap(material->textureCutout, texcoord.x, texcoord.y));
}

/* optixTrace of a radiance ray (raygeneration.cu:84-89) with the radiance any-hit program applied in canonical order */
static int trace_radiance(const shade_ctx* c, const float o[3], const float d[3], float tmin, float tmax, besthit* hit, uint32_t* seed)
{
  const orc_scene* s = c->s;
  if (!s->hasCutout) return trace_scene(s, o, d, tmin, tmax, c->mode, 0, hit, c->st);
  hitkey skip; const hitkey* after = NULL;
  for (;;)
  {
    if (!trace_scene_after(s, o, d, tmin, tmax, c->mode, 0, hit, c->st, after)) return 0;
    const rt_MaterialDefinition* material = &s->materials[s->insts[hit->inst].material];
    if (material->textureCutout == 0) return 1;                      /* hit records without an any-hit program */
    const float opacity = cutout_opacity(s, material, hit);
    if (opacity < 1.0f && opacity <= orc_rng(seed)) { skip.t = hit->t; skip.inst = hit->inst; skip.prim = hit->prim; after = &skip; continue; }
    return 1;
  }
}

/* optixTrace of a shadow ray (closesthit.cu:281-286): __anyhit__shadow terminates at any candidate, __anyhit__shadow_cutout
 * ignores it stochastically.  Returns 1 when the visibility test failed (FLAG_SHADOW). */
static int trace_shadow(const shade_ctx* c, const float o[3], const float d[3], float tmin, float tmax, uint32_t* seed)
{
  const orc_scene* s = c->s;
  besthit hit;
  if (!s->hasCutout) return trace_scene(s, o, d, tmin, tmax, c->mode, 1, &hit, c->st);
  hitkey skip; const hitkey* after = NULL;
  for (;;)
  {
    if (!trace_scene_after(s, o, d, tmin, tmax, c->mode, 0, &hit, c->st, after)) return 0;
    const rt_MaterialDefinition* material = &s->materials[s->insts[hit.inst].material];
    if (material->textureCutout == 0) return 1;
    const float opacity = cutout_opacity(s, material, &hit);
    if (opacity < 1.0f && opacity <= orc_rng(seed)) { skip.t = hit.t; skip.inst = hit.inst; skip.prim = hit.prim; after = &skip; continue; }
    return 1;
  }
}

static void closest_hit(const shade_ctx* c, const besthit* hit, prd_t* prd)
{
  const orc_scene* s = c->s;
  const instance* in = &s->insts[hit->inst];
  const geometry* g = &s->geoms[in->geometry];
  const uint32_t* tri = &g->indices[3u * hit->prim];
  const rt_TriangleAttributes* a0 = &g->attrs[tri[0]];
  const rt_TriangleAttributes* a1 = &g->attrs[tri[1]];
  const rt_TriangleAttributes* a2 = &g->attrs[tri[2]];
  const float bx = hit->u, by = hit->v;
  const float alpha = 1.0f - bx - by;

  const v3 ng = vcross(vsub(from_f3(a1->vertex), from_f3(a0->vertex)), vsub(from_f3(a2->vertex), from_f3(a0->vertex)));
  const v3 tg = vadd(vadd(vscale(from_f3(a0->tangent), alpha), vscale(from_f3(a1->tangent), bx)), vscale(from_f3(a2->tangent), by));
  const v3 ns = vadd(vadd(vscale(from_f3(a0->normal), alpha), vscale(from_f3(a1->normal), bx)), vscale(from_f3(a2->normal), by));

  state_t state;
  state.texcoord = vadd(vadd(vscale(from_f3(a0->texcoord), alpha), vscale(from_f3(a1->texcoord), bx)), vscale(from_f3(a2->texcoord), by));
  state.normalGeo = vnormalize(xf_normal(in->inv, ng));
  state.tangent   = vnormalize(xf_vector(in->m, tg));
  state.normal    = vnormalize(xf_normal(in->inv, ns));

  prd->distance = hit->t;
  prd->pos = vadd(prd->pos, vscale(prd->wi, prd->distance));
  prd->flags |= (0.0f <= vdot(prd->wo, state.normalGeo)) ? RT_FLAG_FRONTFACE : 0u;
  if ((prd->flags & RT_FLAG_FRONTFACE) == 0)
  {
    state.normalGeo = vneg(state.normalGeo);
    state.tangent = vneg(state.tangent);
    state.normal = vneg(state.normal);
  }
  prd->radiance = v3s(0.0f);

  if (0 <= in->light && (prd->flags & RT_FLAG_FRONTFACE))
  {
    const float cosTheta = vdot(prd->wo, state.normalGeo);
    if (RT_DENOMINATOR_EPSILON < cosTheta)
    {
      const rt_LightDefinition* light = &s->lights[in->light];
      v3 emission = from_f3(light->emission);
      const float lightPdf = (prd->distance * prd->distance) / (light->area * cosTheta);
      if ((prd->flags & RT_FLAG_DIFFUSE) && RT_DENOMINATOR_EPSILON < lightPdf)
        emission = vscale(emission, power_heuristic(prd->pdf, lightPdf));
      prd->radiance = emission;
      prd->flags |= RT_FLAG_TERMINATE;
      return;
    }
  }

  prd->f_over_pdf = v3s(0.0f);
  prd->pdf = 0.0f;
  const rt_MaterialDefinition* material = &s->materials[in->material];
  state.albedo = from_f3(material->albedo);
  if (material->textureAlbedo != 0)   /* closesthit.cu:233-240 */
    state.albedo = vmul(state.albedo, tex2d_wrap(material->textureAlbedo, state.texcoord.x, state.texcoord.y));
  prd->flags = (prd->flags & ~RT_FLAG_DIFFUSE) | RT_FLAG_HIT | material->flags;
  bsdf_sample(material, &state, prd);

  const int numLights = c->sys->numLights;
  if ((prd->flags & RT_FLAG_DIFFUSE) && 0 < numLights)
  {
    const v2 sample = rng2(&prd->seed);
    light_sample_t ls; memset(&ls, 0, sizeof(ls));
    if (1 < numLights)
    {
      int idx = (int)floorf(orc_rng(&prd->seed) * (float)numLights);
      if (idx < 0) idx = 0; if (idx > numLights - 1) idx = numLights - 1;
      ls.index = idx;
    }
    else ls.index = 0;
    const int type = s->lights[ls.index].type;
    if (type == RT_LIGHT_PARALLELOGRAM) light_parallelogram(s, numLights, prd->pos, sample, &ls);
    else if (c->miss == RT_MISS_SPHERE) light_env_sphere(s, numLights, c->sys->envRotation, prd->pos, sample, &ls);
    else                                light_env_constant(s, numLights, prd->pos, sample, &ls);
    if (0.0f < ls.pdf)
    {
      const v4 bp = bsdf_eval(material, &state, prd, ls.direction);
      const v3 f = V3(bp.x, bp.y, bp.z);
      if (0.0f < bp.w && !v3_is_null(f))
      {
        const float o[3] = { prd->pos.x, prd->pos.y, prd->pos.z }, d[3] = { ls.direction.x, ls.direction.y, ls.direction.z };
        if (c->st) c->st->shadowRays++;
        const int occluded = trace_shadow(c, o, d, c->sys->sceneEpsilon, ls.distance - c->sys->sceneEpsilon, &prd->seed);
        if (!occluded)
        {
          if (prd->flags & RT_FLAG_VOLUME)
          {
            const v3 e = V3(rt_expf(-ls.distance * prd->sigma_t.x), rt_expf(-ls.distance * prd->sigma_t.y), rt_expf(-ls.distance * prd->sigma_t.z));
            ls.emission = vmul(ls.emission, e);
          }
          const float weightMis = power_heuristic(ls.pdf, bp.w);
          prd->radiance = vadd(prd->radiance, vscale(vmul(f, ls.emission), weightMis * vdot(ls.direction, state.normal) / ls.pdf));
        }
      }
    }
  }
}

/* ---- integrator (raygeneration.cu:42-149) ---- */
static v3 integrator(const shade_ctx* c, prd_t* prd)
{
  v4 stack[RT_MATERIAL_STACK_SIZE];
  int stackIdx = RT_MATERIAL_STACK_EMPTY;
  int depth = 0;
  v3 radiance = v3s(0.0f), throughput = v3s(1.0f);
  prd->absorption_ior.x = 0.0f; prd->absorption_ior.y = 0.0f; prd->absorption_ior.z = 0.0f; prd->absorption_ior.w = 1.0f;
  prd->sigma_t = v3s(0.0f);
  prd->flags = 0;
  prd->pdf = 0.0f;               /* uninitialised in the reference; never read before the first hit writes it */
  prd->f_over_pdf = v3s(0.0f);
  memset(stack, 0, sizeof(stack));

  while (depth < c->sys->pathLengths.y)
  {
    prd->wo = vneg(prd->wi);
    prd->ior.x = 1.0f; prd->ior.y = 1.0f;
    prd->distance = RT_DEFAULT_MAX;
    prd->flags &= RT_FLAG_CLEAR_MASK;
    if (RT_MATERIAL_STACK_FIRST <= stackIdx)
    {
      prd->flags |= RT_FLAG_VOLUME;
      prd->sigma_t = V3(stack[stackIdx].x, stack[stackIdx].y, stack[stackIdx].z);
      prd->ior.x = stack[stackIdx].w;
      if (RT_MATERIAL_STACK_FIRST <= stackIdx - 1) prd->ior.y = stack[stackIdx - 1].w;
    }

    const float o[3] = { prd->pos.x, prd->pos.y, prd->pos.z }, d[3] = { prd->wi.x, prd->wi.y, prd->wi.z };
    besthit hit;
    if (c->st) c->st->radianceRays++;
    if (trace_radiance(c, o, d, c->sys->sceneEpsilon, prd->distance, &hit, &prd->seed)) closest_hit(c, &hit, prd);
    else miss_program(c->s, c->miss, c->sys->envRotation, prd);

    if (prd->flags & RT_FLAG_VOLUME)
    {
      const v3 e = V3(rt_expf(-prd->distance * prd->sigma_t.x), rt_expf(-prd->distance * prd->sigma_t.y), rt_expf(-prd->distance * prd->sigma_t.z));
      throughput = vmul(throughput, e);
    }
    radiance = vadd(radiance, vmul(throughput, prd->radiance));
    if ((prd->flags & RT_FLAG_TERMINATE) || prd->pdf <= 0.0f || v3_is_null(prd->f_over_pdf)) break;
    throughput = vmul(throughput, prd->f_over_pdf);
    if (c->sys->pathLengths.x <= depth)
    {
      const float probability = fmax3(throughput);
      if (probability < orc_rng(&prd->seed)) break;
      throughput = vdivs(throughput, probability);
    }
    if ((prd->flags & (RT_FLAG_THINWALLED | RT_FLAG_TRANSMISSION)) == RT_FLAG_TRANSMISSION)
    {
      if (prd->flags & RT_FLAG_FRONTFACE)
      {
        stackIdx = (stackIdx + 1 < RT_MATERIAL_STACK_LAST) ? stackIdx + 1 : RT_MATERIAL_STACK_LAST;
        stack[stackIdx] = prd->absorption_ior;
      }
      else
      {
        stackIdx = (stackIdx - 1 > RT_MATERIAL_STACK_EMPTY) ? stackIdx - 1 : RT_MATERIAL_STACK_EMPTY;
      }
    }
    ++depth;
  }
  return radiance;
}

/* raygeneration.cu:152-164 */
static inline uint32_t distribute(const rt_SystemData* sys, uint32_t x, uint32_t y)
{
  const uint32_t xBlock = x >> sys->tileShift.x;
  const uint32_t yBlock = y >> sys->tileShift.y;
  const uint32_t xTile = xBlock * (uint32_t)sys->deviceCount + (((uint32_t)sys->deviceIndex + yBlock) % (uint32_t)sys->deviceCount);
  return xTile * (uint32_t)sys->tileSize.x + (x & (uint32_t)(sys->tileSize.x - 1));
}

/* raygeneration.cu:173-201: returns 0 when the launch index maps outside the image */
static int start_path(const orc_scene* s, const rt_SystemData* sys, uint32_t launchWidth, uint32_t x, uint32_t y, int iteration,
                      prd_t* prd, uint32_t* column)
{
  uint32_t col = x;
  if (sys->distribution && 1 < sys->deviceCount)
  {
    col = distribute(sys, x, y);
    if ((uint32_t)sys->resolution.x <= col) return 0;
  }
  const uint32_t seedIndex = launchWidth * y + col * (uint32_t)sys->deviceCount + (uint32_t)sys->deviceIndex;
  prd->seed = orc_tea4(seedIndex, (uint32_t)iteration);
  const v2 screen = { (float)sys->resolution.x, (float)sys->resolution.y };
  const v2 pixel = { (float)col, (float)y };
  const v2 sample = rng2(&prd->seed);
  lens_shader(s, sys->lensShader, screen, pixel, sample, &prd->pos, &prd->wi);
  *column = col;
  return 1;
}

void orc_generate_primary(const orc_scene* s, const rt_SystemData* sys, uint32_t launchWidth, uint32_t launchHeight,
                          int iteration, orc_ray* rays)
{
  for (uint32_t y = 0; y < launchHeight; ++y)
    for (uint32_t x = 0; x < launchWidth; ++x)
    {
      orc_ray* r = &rays[(size_t)y * launchWidth + x];
      prd_t prd; uint32_t col;
      memset(&prd, 0, sizeof(prd));
      if (!start_path(s, sys, launchWidth, x, y, iteration, &prd, &col))
      {
        memset(r, 0, sizeof(*r)); r->tmax = -1.0f;
        continue;
      }
      r->ox = prd.pos.x; r->oy = prd.pos.y; r->oz = prd.pos.z; r->tmin = sys->sceneEpsilon;
      r->dx = prd.wi.x;  r->dy = prd.wi.y;  r->dz = prd.wi.z;  r->tmax = RT_DEFAULT_MAX;
    }
}

typedef struct {
  const orc_scene* s; const rt_SystemData* sys; int miss; uint32_t launchWidth, launchHeight; int localCopy;
  int iterFirst, iterCount, rowStep, rowOffset; float* buffer;
  int threadIndex, threadCount; orc_stats stats;
} render_job;

static void* render_worker(void* arg)
{
  render_job* j = (render_job*)arg;
  shade_ctx c = { j->s, j->sys, j->miss, 0, &j->stats };
  uint32_t rowCounter = 0;
  for (uint32_t y = 0; y < j->launchHeight; ++y)
  {
    if ((int)(y % (uint32_t)j->rowStep) != j->rowOffset) continue;
    if ((int)(rowCounter++ % (uint32_t)j->threadCount) != j->threadIndex) continue;
    for (uint32_t x = 0; x < j->launchWidth; ++x)
    {
      for (int it = j->iterFirst; it < j->iterFirst + j->iterCount; ++it)
      {
        prd_t prd; uint32_t col;
        memset(&prd, 0, sizeof(prd));
        if (!start_path(j->s, j->sys, j->launchWidth, x, y, it, &prd, &col)) break;
        v3 radiance = integrator(&c, &prd);
        j->stats.pathSamples++;
        if (!(isnan(radiance.x) || isnan(radiance.y) || isnan(radiance.z)))
        {
          const size_t index = j->localCopy ? ((size_t)y * j->launchWidth + x) : ((size_t)y * (size_t)j->sys->resolution.x + col);
          float* dst = &j->buffer[4 * index];
          if (0 < it)
          {
            /* lerp(dst, radiance, 1/(it+1)) = dst + t*(radiance - dst), raygeneration.cu:248-250 */
            const float t = 1.0f / (float)(it + 1);
            radiance = V3(dst[0] + t * (radiance.x - dst[0]), dst[1] + t * (radiance.y - dst[1]), dst[2] + t * (radiance.z - dst[2]));
          }
          dst[0] = radiance.x; dst[1] = radiance.y; dst[2] = radiance.z; dst[3] = 1.0f;
        }
      }
    }
  }
  return NULL;
}

static void stats_add(orc_stats* a, const orc_stats* b)
{
  a->radianceRays += b->radianceRays; a->shadowRays += b->shadowRays; a->pathSamples += b->pathSamples;
  a->nodesVisited += b->nodesVisited; a->trisTested += b->trisTested; a->instancesEntered += b->instancesEntered;
}

void orc_render(const orc_scene* s, const rt_SystemData* sys, int miss, uint32_t launchWidth, uint32_t launchHeight,
                int localCopy, int iterFirst, int iterCount, int rowStep, int rowOffset, int threads,
                float* buffer, orc_stats* stats)
{
  if (threads <= 0) threads = orc_online_cores();
  if (threads > 256) threads = 256;
  if (rowStep < 1) rowStep = 1;
  render_job jobs[256]; pthread_t tids[256];
  for (int t = 0; t < threads; ++t)
  {
    render_job* j = &jobs[t];
    memset(j, 0, sizeof(*j));
    j->s = s; j->sys = sys; j->miss = miss; j->launchWidth = launchWidth; j->launchHeight = launchHeight; j->localCopy = localCopy;
    j->iterFirst = iterFirst; j->iterCount = iterCount; j->rowStep = rowStep; j->rowOffset = rowOffset; j->buffer = buffer;
    j->threadIndex = t; j->threadCount = threads;
    if (threads > 1) pthread_create(&tids[t], NULL, render_worker, j);
    else render_worker(j);
  }
  for (int t = 0; t < threads; ++t)
  {
    if (threads > 1) pthread_join(tids[t], NULL);
    if (stats) stats_add(stats, &jobs[t].stats);
  }
}

void orc_path_radiance(const orc_scene* s, const rt_SystemData* sys, int miss, uint32_t launchWidth,
                       const uint32_t* launchXY, uint64_t n, int iteration, float* out, orc_stats* stats)
{
  orc_stats local; memset(&local, 0, sizeof(local));
  shade_ctx c = { s, sys, miss, 0, &local };
  for (uint64_t i = 0; i < n; ++i)
  {
    prd_t prd; uint32_t col;
    memset(&prd, 0, sizeof(prd));
    v3 L = v3s(0.0f);
    if (start_path(s, sys, launchWidth, launchXY[2 * i], launchXY[2 * i + 1], iteration, &prd, &col)) { L = integrator(&c, &prd); local.pathSamples++; }
    out[3 * i] = L.x; out[3 * i + 1] = L.y; out[3 * i + 2] = L.z;
  }
  if (stats) stats_add(stats, &local);
}

/* shaders/compositor.cu:38-65 */
void orc_composite(const rt_CompositorData* a, const float* tileBuffer, float* outputBuffer)
{
  for (int y = 0; y < a->resolution.y; ++y)
    for (int x = 0; x < a->launchWidth; ++x)
    {
      const uint32_t xBlock = (uint32_t)x >> a->tileShift.x, yBlock = (uint32_t)y >> a->tileShift.y;
      const uint32_t xTile = xBlock * (uint32_t)a->deviceCount + (((uint32_t)a->deviceIndex + yBlock) % (uint32_t)a->deviceCount);
      const uint32_t xPixel = xTile * (uint32_t)a->tileSize.x + ((uint32_t)x & (uint32_t)(a->tileSize.x - 1));
      if (xPixel < (uint32_t)a->resolution.x)
        memcpy(&outputBuffer[4 * ((size_t)y * (size_t)a->resolution.x + xPixel)], &tileBuffer[4 * ((size_t)y * (size_t)a->launchWidth + (size_t)x)], sizeof(float) * 4);
    }
}

/* src/Application.cpp:2262-2295 */
void orc_tonemap(const rt_TonemapperParams* p, const float* rgba, uint8_t* rgb, uint64_t numPixels)
{
  const float invGamma = 1.0f / p->gamma;
  const v3 colorBalance = V3(p->colorBalance[0], p->colorBalance[1], p->colorBalance[2]);
  const float invWhitePoint = p->brightness / p->whitePoint;
  const float burnHighlights = p->burnHighlights;
  const float crushBlacks = p->crushBlacks + p->crushBlacks + 1.0f;
  const float saturation = p->saturation;
  const v3 lumw = V3(0.3f, 0.59f, 0.11f);
  for (uint64_t i = 0; i < numPixels; ++i)
  {
    const v3 hdr = V3(rgba[4 * i], rgba[4 * i + 1], rgba[4 * i + 2]);
    v3 ldr = vmul(vscale(colorBalance, invWhitePoint), hdr);
    const v3 num = vadd(vscale(ldr, burnHighlights), v3s(1.0f)), den = vadd(ldr, v3s(1.0f));
    ldr = vmul(ldr, V3(num.x / den.x, num.y / den.y, num.z / den.z));
    float lum = vdot(ldr, lumw);
    ldr = vadd(v3s(lum), vscale(vsub(ldr, v3s(lum)), saturation));
    ldr = V3(fmaxf(0.0f, ldr.x), fmaxf(0.0f, ldr.y), fmaxf(0.0f, ldr.z));
    lum = vdot(ldr, lumw);
    if (lum < 1.0f)
    {
      const v3 crushed = V3(rt_powf(ldr.x, crushBlacks), rt_powf(ldr.y, crushBlacks), rt_powf(ldr.z, crushBlacks));
      ldr = vadd(crushed, vscale(vsub(ldr, crushed), sqrtf(lum)));
      ldr = V3(fmaxf(0.0f, ldr.x), fmaxf(0.0f, ldr.y), fmaxf(0.0f, ldr.z));
    }
    float c[3] = { rt_powf(ldr.x, invGamma), rt_powf(ldr.y, invGamma), rt_powf(ldr.z, invGamma) };
    for (int k = 0; k < 3; ++k)
    {
      if (c[k] < 0.0f) c[k] = 0.0f; if (c[k] > 1.0f) c[k] = 1.0f;
      rgb[3 * i + k] = (uint8_t)(c[k] * 255.0f);
    }
  }
}

/* ------------------------------------------------------------------------------------------
 * TEST HOOKS: function-level access to the BSDF and light restatements above.  tests/test_cpu_shade_source.py compares the
 * PRODUCT's csrc/shade.cuh, compiled for the host, with them word for word.  prd = the 28 words of prd_t in declaration order
 * (pos 0-2, distance 3, wo 4-6, wi 7-9, radiance 10-12, flags 13, f_over_pdf 14-16, pdf 17, sigma_t 18-20, ior 21-22,
 * absorption_ior 23-26, seed 27); st = normalGeo, tangent, normal, albedo (12 floats); light out = direction, distance,
 * emission, pdf (8 floats).
 * ------------------------------------------------------------------------------------------ */
static void prd_unpack(prd_t* p, const uint32_t w[28])
{
  float f[28]; memcpy(f, w, sizeof(f));
  p->pos = (v3){ f[0], f[1], f[2] }; p->distance = f[3];
  p->wo = (v3){ f[4], f[5], f[6] }; p->wi = (v3){ f[7], f[8], f[9] };
  p->radiance = (v3){ f[10], f[11], f[12] }; p->flags = w[13];
  p->f_over_pdf = (v3){ f[14], f[15], f[16] }; p->pdf = f[17];
  p->sigma_t = (v3){ f[18], f[19], f[20] }; p->ior = (v2){ f[21], f[22] };
  p->absorption_ior = (v4){ f[23], f[24], f[25], f[26] }; p->seed = w[27];
}

static void prd_pack(const prd_t* p, uint32_t w[28])
{
  const float f[28] = { p->pos.x, p->pos.y, p->pos.z, p->distance, p->wo.x, p->wo.y, p->wo.z, p->wi.x, p->wi.y, p->wi.z,
                        p->radiance.x, p->radiance.y, p->radiance.z, 0.0f, p->f_over_pdf.x, p->f_over_pdf.y, p->f_over_pdf.z, p->pdf,
                        p->sigma_t.x, p->sigma_t.y, p->sigma_t.z, p->ior.x, p->ior.y,
                        p->absorption_ior.x, p->absorption_ior.y, p->absorption_ior.z, p->absorption_ior.w, 0.0f };
  memcpy(w, f, sizeof(f));
  w[13] = p->flags; w[27] = p->seed;
}

static state_t state_unpack(const float st[12])
{
  state_t s;
  s.normalGeo = (v3){ st[0], st[1], st[2] }; s.tangent = (v3){ st[3], st[4], st[5] }; s.normal = (v3){ st[6], st[7], st[8] };
  s.texcoord = (v3){ 0.0f, 0.0f, 0.0f }; s.albedo = (v3){ st[9], st[10], st[11] };
  return s;
}

void orc_test_bsdf_sample(const rt_MaterialDefinition* m, const float st[12], uint32_t prd[28])
{
  const state_t s = state_unpack(st);
  prd_t p; prd_unpack(&p, prd);
  bsdf_sample(m, &s, &p);
  prd_pack(&p, prd);
}

void orc_test_bsdf_eval(const rt_MaterialDefinition* m, const float st[12], const uint32_t prd[28], const float wiL[3], float out[4])
{
  const state_t s = state_unpack(st);
  prd_t p; prd_unpack(&p, prd);
  const v4 r = bsdf_eval(m, &s, &p, (v3){ wiL[0], wiL[1], wiL[2] });
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

static void light_pack(const light_sample_t* ls, float out[8])
{
  out[0] = ls->direction.x; out[1] = ls->direction.y; out[2] = ls->direction.z; out[3] = ls->distance;
  out[4] = ls->emission.x; out[5] = ls->emission.y; out[6] = ls->emission.z; out[7] = ls->pdf;
}

void orc_test_light_constant(int numLights, const float sample[2], float out[8])
{
  light_sample_t ls; memset(&ls, 0, sizeof(ls));
  light_env_constant(NULL, numLights, (v3){ 0.0f, 0.0f, 0.0f }, (v2){ sample[0], sample[1] }, &ls);
  light_pack(&ls, out);
}

void orc_test_light_parallelogram(const rt_LightDefinition* light, int numLights, const float point[3], const float sample[2], float out[8])
{
  orc_scene tmp; memset(&tmp, 0, sizeof(tmp));
  tmp.lights = (rt_LightDefinition*)light; tmp.numLightDefs = 1;
  light_sample_t ls; memset(&ls, 0, sizeof(ls));
  ls.index = 0;
  light_parallelogram(&tmp, numLights, (v3){ point[0], point[1], point[2] }, (v2){ sample[0], sample[1] }, &ls);
  light_pack(&ls, out);
}

/* env: RGBA32F texels (w x h), the two CDF tables of the environment light, integral, rotation */
static void env_scene(orc_scene* tmp, const float* texels, uint32_t w, uint32_t h, const float* cdfU, const float* cdfV, float integral)
{
  memset(tmp, 0, sizeof(*tmp));
  tmp->envTexels = (float*)texels; tmp->envW = w; tmp->envH = h;
  tmp->envCdfU = (float*)cdfU; tmp->envCdfV = (float*)cdfV; tmp->envIntegral = integral;
}

void orc_test_miss(const float* texels, uint32_t w, uint32_t h, float integral, float rotation, int miss, uint32_t prd[28])
{
  orc_scene tmp; env_scene(&tmp, texels, w, h, NULL, NULL, integral);
  prd_t p; prd_unpack(&p, prd);
  miss_program(&tmp, miss, rotation, &p);
  prd_pack(&p, prd);
}

void orc_test_light_sphere(const float* texels, uint32_t w, uint32_t h, const float* cdfU, const float* cdfV, float integral, float rotation,
                           int numLights, const float sample[2], float out[8])
{
  orc_scene tmp; env_scene(&tmp, texels, w, h, cdfU, cdfV, integral);
  light_sample_t ls; memset(&ls, 0, sizeof(ls));
  light_env_sphere(&tmp, numLights, rotation, (v3){ 0.0f, 0.0f, 0.0f }, (v2){ sample[0], sample[1] }, &ls);
  light_pack(&ls, out);
}

#include "wide_bvh.inc"
