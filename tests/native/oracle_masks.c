/* tests/native/oracle_masks.c -- TEST INFRASTRUCTURE: the scalar oracle extended by the visibility masks and face culling of
 * rtc_trace_closest_ex / rtc_trace_any_ex / rtc_trace_count_ex.
 *
 * oracle/rt_oracle.c (and the oracle/wide_bvh.inc it includes) is included here unchanged, so this file uses the oracle's own
 * scene, object-space ray, vertex fetch, tie rule and wide-BVH box test.  It adds:
 *   - mk_trace_closest / mk_trace_any: brute force over every triangle of every instance whose mask shares a bit with the ray
 *     mask.  mode 1 decides facing as the kernels do, by the sign of the watertight test's det (det > 0 is front-facing;
 *     DESIGN.md section 3 derives it).  mode 0 restates the geometric definition instead: front-facing when
 *     dot((v1 - v0) x (v2 - v0), d) < 0 in double, d the object-space direction.
 *   - mk_wide_trace: oracle/wide_bvh.inc's w_trace_one with the two tests in the places the FILTER traversal of
 *     csrc/trace.cuh has them (a masked-out instance is skipped before it is entered and is not counted; a culled candidate is
 *     no hit), so that the counters of rtc_trace_count_ex are reproduced ray by ray.
 * cullFlags: bit 0 culls back-facing, bit 1 front-facing candidates (RTC_RAY_CULL_*).
 */
#include "rt_oracle.c"

/* the oracle's tri_test, with det as an output (the same operations in the same order) */
static int mk_tri_test_det(const oray* r, const float* v0, const float* v1, const float* v2, float* t, float* beta, float* gamma,
                           float* detOut)
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
  *detOut = det;
  return 1;
}

static int mk_culled_by_det(uint32_t cullFlags, float det)
{
  return (cullFlags & (det > 0.0f ? 2u : 1u)) != 0u;
}

static int mk_culled_by_normal(uint32_t cullFlags, const oray* r, const float* v0, const float* v1, const float* v2)
{
  const double e1[3] = { (double)v1[0] - v0[0], (double)v1[1] - v0[1], (double)v1[2] - v0[2] };
  const double e2[3] = { (double)v2[0] - v0[0], (double)v2[1] - v0[1], (double)v2[2] - v0[2] };
  const double n[3] = { e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0] };
  const double dn = n[0] * r->d[0] + n[1] * r->d[1] + n[2] * r->d[2];
  return (cullFlags & (dn < 0.0 ? 2u : 1u)) != 0u;
}

/* one ray by brute force; returns 1 on a hit (any hit: the first one) */
static int mk_trace_one(const orc_scene* s, const uint8_t* masks, uint32_t rayMask, uint32_t cullFlags, int mode, const orc_ray* ray,
                        int anyHit, besthit* best)
{
  const float o[3] = { ray->ox, ray->oy, ray->oz }, d[3] = { ray->dx, ray->dy, ray->dz };
  const float tmin = ray->tmin, tmax = ray->tmax;
  best->inst = 0xffffffffu; best->prim = 0xffffffffu; best->t = -1.0f; best->u = 0.0f; best->v = 0.0f; best->skip = NULL;
  if (!(tmax > tmin)) return 0;
  for (int ii = 0; ii < s->numInsts; ++ii)
  {
    const instance* in = &s->insts[ii];
    const geometry* g = &s->geoms[in->geometry];
    if (g->numTris == 0 || !in->active || !(masks[ii] & rayMask)) continue;
    oray r; to_object(in->inv, o, d, &r);
    for (uint32_t p = 0; p < g->numTris; ++p)
    {
      if (!tri_active(g, p)) continue;
      const float *v0, *v1, *v2; float t, u, v, det;
      tri_verts(g, p, &v0, &v1, &v2);
      if (!mk_tri_test_det(&r, v0, v1, v2, &t, &u, &v, &det)) continue;
      if (mode ? mk_culled_by_det(cullFlags, det) : mk_culled_by_normal(cullFlags, &r, v0, v1, v2)) continue;
      if (anyHit) { if (t > tmin && t < tmax) return 1; }
      else consider(best, t, u, v, (uint32_t)ii, p, tmin, tmax);
    }
  }
  return !anyHit && best->inst != 0xffffffffu;
}

/* masks: one byte per instance of the scene */
void mk_trace_closest(const orc_scene* s, const uint8_t* masks, uint32_t rayMask, uint32_t cullFlags, int mode, const orc_ray* rays,
                      uint64_t n, orc_hit* hits)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    besthit b;
    mk_trace_one(s, masks, rayMask, cullFlags, mode, rays + i, 0, &b);
    hits[i].t = b.t; hits[i].u = b.u; hits[i].v = b.v; hits[i].inst = b.inst; hits[i].prim = b.prim;
  }
}

void mk_trace_any(const orc_scene* s, const uint8_t* masks, uint32_t rayMask, uint32_t cullFlags, int mode, const orc_ray* rays,
                  uint64_t n, uint8_t* occluded)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    besthit b;
    occluded[i] = (uint8_t)mk_trace_one(s, masks, rayMask, cullFlags, mode, rays + i, 1, &b);
  }
}

/* oracle/wide_bvh.inc w_trace_one with the FILTER tests of csrc/trace.cuh; counts: [0] nodes, [1] triangles, [2] instances */
static void mk_w_trace_one(const orc_wide_scene* ws, const orc_ray* ray, int any, const uint8_t* masks, uint32_t rayMask,
                           uint32_t cullFlags, orc_hit* hit, uint64_t counts[3])
{
  hit->t = -1.0f; hit->u = 0.0f; hit->v = 0.0f; hit->inst = 0xffffffffu; hit->prim = 0xffffffffu;
  const float tmin = ray->tmin;
  float tlimit = ray->tmax;
  if (!(tlimit > tmin)) return;
  uint32_t stack[W_STACK][2];
  int sp = 0, blasBase = -1;
  uint32_t curInst = 0;
  wbox br;
  w_box_setup(&br, ray->ox, ray->oy, ray->oz, ray->dx, ray->dy, ray->dz);
  oray orr;
  memset(&orr, 0, sizeof(orr));
  const orc_wnode* nodes = ws->tlasNodes;
  const float* tris = NULL;
  uint32_t ngx = 0u, ngy = 0x80000000u, tgx = 0u, tgy = 0u;
  for (;;)
  {
    if (ngy & 0xff000000u)
    {
      uint32_t bit = 31u; while (!((ngy >> bit) & 1u)) --bit;
      ngy &= ~(1u << bit);
      if (ngy & 0xff000000u) { stack[sp][0] = ngx; stack[sp][1] = ngy; ++sp; }
      const uint32_t slot = (bit - 24u) ^ br.octinv;
      const uint32_t rel = (uint32_t)__builtin_popcount(ngy & 0xffu & ((1u << slot) - 1u));
      const orc_wnode* n = nodes + (ngx + rel);
      counts[0]++;
      const uint32_t hits = w_node_test(&br, n, tmin, tlimit);
      const uint32_t imask = n->imask;
      ngx = n->childBase; ngy = (w_xor_permute8(hits & imask, br.octinv) << 24) | imask;
      uint32_t leaf = hits & ~imask & 0xffu, primMask = 0u;
      while (leaf)
      {
        const uint32_t s = (uint32_t)__builtin_ctz(leaf);
        leaf &= leaf - 1u;
        const uint32_t meta = n->meta[s];
        primMask |= ((1u << (meta >> 5)) - 1u) << (meta & 31u);
      }
      tgx = n->triBase; tgy = primMask;
    }
    else { tgx = ngx; tgy = ngy; ngx = 0u; ngy = 0u; }

    int done = 0;
    while (tgy)
    {
      const uint32_t idx = (uint32_t)__builtin_ctz(tgy);
      tgy &= tgy - 1u;
      if (blasBase < 0)
      {
        const uint32_t inst = ws->tlasLeaves[tgx + idx];
        if (!(masks[inst] & rayMask)) continue;                 /* masked out: not entered, next leaf bit */
        if (tgy) { stack[sp][0] = tgx; stack[sp][1] = tgy; ++sp; }
        if (ngy & 0xff000000u) { stack[sp][0] = ngx; stack[sp][1] = ngy; ++sp; }
        counts[2]++;
        const float* m = ws->worldToObject + 12u * (size_t)inst;
        orr.o[0] = fmaf(m[0], ray->ox, fmaf(m[1], ray->oy, fmaf(m[2], ray->oz, m[3])));
        orr.o[1] = fmaf(m[4], ray->ox, fmaf(m[5], ray->oy, fmaf(m[6], ray->oz, m[7])));
        orr.o[2] = fmaf(m[8], ray->ox, fmaf(m[9], ray->oy, fmaf(m[10], ray->oz, m[11])));
        orr.d[0] = fmaf(m[0], ray->dx, fmaf(m[1], ray->dy, m[2] * ray->dz));
        orr.d[1] = fmaf(m[4], ray->dx, fmaf(m[5], ray->dy, m[6] * ray->dz));
        orr.d[2] = fmaf(m[8], ray->dx, fmaf(m[9], ray->dy, m[10] * ray->dz));
        oray_setup(&orr);
        w_box_setup(&br, orr.o[0], orr.o[1], orr.o[2], orr.d[0], orr.d[1], orr.d[2]);
        curInst = inst;
        blasBase = sp;
        nodes = ws->gasNodes[ws->instGas[inst]];
        tris = ws->gasTris[ws->instGas[inst]];
        ngx = 0u; ngy = 0x80000000u; tgx = 0u; tgy = 0u;
        break;
      }
      else
      {
        const float* tp = tris + 12u * (size_t)(tgx + idx);
        counts[1]++;
        float t, beta, gamma, det;
        if (mk_tri_test_det(&orr, tp, tp + 4, tp + 8, &t, &beta, &gamma, &det) && !mk_culled_by_det(cullFlags, det) && t > tmin)
        {
          uint32_t prim; memcpy(&prim, tp + 3, 4);
          if (any)
          {
            if (t < tlimit) { hit->t = t; hit->inst = curInst; hit->prim = prim; done = 1; break; }
          }
          else
          {
            const int better = (hit->inst != 0xffffffffu) ? (t < hit->t || (t == hit->t && (curInst < hit->inst || (curInst == hit->inst && prim < hit->prim))))
                                                          : (t < tlimit);
            if (better) { tlimit = t; hit->t = t; hit->inst = curInst; hit->prim = prim; hit->u = beta; hit->v = gamma; }
          }
        }
      }
    }
    if (done) return;
    if (!(ngy & 0xff000000u))
    {
      if (blasBase >= 0 && sp == blasBase)
      {
        blasBase = -1;
        nodes = ws->tlasNodes;
        w_box_setup(&br, ray->ox, ray->oy, ray->oz, ray->dx, ray->dy, ray->dz);
      }
      if (sp == 0) return;
      --sp; ngx = stack[sp][0]; ngy = stack[sp][1];
    }
  }
}

void mk_wide_trace(const orc_wide_scene* ws, const orc_ray* rays, uint64_t n, int any, const uint8_t* masks, uint32_t rayMask,
                   uint32_t cullFlags, orc_hit* hits, uint64_t counts[3])
{
  counts[0] = counts[1] = counts[2] = 0;
  for (uint64_t i = 0; i < n; ++i)
  {
    orc_hit h;
    mk_w_trace_one(ws, rays + i, any, masks, rayMask, cullFlags, &h, counts);
    if (hits) hits[i] = h;
  }
}
