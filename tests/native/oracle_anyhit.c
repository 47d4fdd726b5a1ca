/* tests/native/oracle_anyhit.c -- TEST INFRASTRUCTURE: brute force for the any-hit callbacks of include/rtc_device.cuh.
 *
 * Built on tests/native/oracle_masks.c (which includes oracle/rt_oracle.c unchanged): the oracle's scene, object-space ray and
 * vertex fetch, mk_tri_test_det and mk_culled_by_det.  A candidate of a ray is a triangle of an instance whose mask shares a bit
 * with the ray's mask, that passes the watertight test and the cull flags, with tmin < t < tmax; u, v are V / det and W / det and
 * frontFacing is det > 0, as the header computes them.  The decisions are those of anyhit_predicates.h.
 *   ah_closest:    the smallest accepted candidate in (t, instance, primitive) order (the oracle's consider())
 *   ah_any:        1 when some candidate is accepted
 *   ah_candidates: every candidate of the ray (in instance, primitive order; the first K are written, counts[i] is the total)
 * rayMasks / rayFlags / p0 / p1: one per ray.
 */
#include "oracle_masks.c"
#include "anyhit_predicates.h"

typedef void (*ah_visit)(void* ctx, const ahp_record* c);

static void ah_each_candidate(const orc_scene* s, const uint8_t* masks, uint32_t rayMask, uint32_t cullFlags, const orc_ray* ray,
                              ah_visit visit, void* ctx)
{
  const float o[3] = { ray->ox, ray->oy, ray->oz }, d[3] = { ray->dx, ray->dy, ray->dz };
  if (!(ray->tmax > ray->tmin)) return;
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
      if (!mk_tri_test_det(&r, v0, v1, v2, &t, &u, &v, &det) || mk_culled_by_det(cullFlags, det)) continue;
      if (!(t > ray->tmin && t < ray->tmax)) continue;
      const ahp_record c = { t, u, v, (uint32_t)ii, p, det > 0.0f ? 1u : 0u };
      visit(ctx, &c);
    }
  }
}

typedef struct { int pred; uint32_t p0, p1; besthit best; int accepted; float tmin, tmax; } ah_decide_ctx;

static void ah_visit_closest(void* vctx, const ahp_record* c)
{
  ah_decide_ctx* x = (ah_decide_ctx*)vctx;
  if (ahp_decide(x->pred, c->t, c->u, c->v, c->inst, c->prim, c->frontFacing, x->p0, x->p1, 0))
    consider(&x->best, c->t, c->u, c->v, c->inst, c->prim, x->tmin, x->tmax);
}

static void ah_visit_any(void* vctx, const ahp_record* c)
{
  ah_decide_ctx* x = (ah_decide_ctx*)vctx;
  if (ahp_decide(x->pred, c->t, c->u, c->v, c->inst, c->prim, c->frontFacing, x->p0, x->p1, 0)) x->accepted = 1;
}

void ah_closest(const orc_scene* s, const uint8_t* masks, const orc_ray* rays, uint64_t n, const uint32_t* rayMasks, const uint32_t* rayFlags,
                int pred, const uint32_t* p0, const uint32_t* p1, orc_hit* hits)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    ah_decide_ctx x;
    x.pred = pred; x.p0 = p0[i]; x.p1 = p1[i]; x.tmin = rays[i].tmin; x.tmax = rays[i].tmax;
    x.best.inst = 0xffffffffu; x.best.prim = 0xffffffffu; x.best.t = -1.0f; x.best.u = 0.0f; x.best.v = 0.0f; x.best.skip = NULL;
    ah_each_candidate(s, masks, rayMasks[i], rayFlags[i], rays + i, ah_visit_closest, &x);
    hits[i].t = x.best.t; hits[i].u = x.best.u; hits[i].v = x.best.v; hits[i].inst = x.best.inst; hits[i].prim = x.best.prim;
  }
}

void ah_any(const orc_scene* s, const uint8_t* masks, const orc_ray* rays, uint64_t n, const uint32_t* rayMasks, const uint32_t* rayFlags,
            int pred, const uint32_t* p0, const uint32_t* p1, uint8_t* occluded)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    ah_decide_ctx x;
    x.pred = pred; x.p0 = p0[i]; x.p1 = p1[i]; x.accepted = 0;
    ah_each_candidate(s, masks, rayMasks[i], rayFlags[i], rays + i, ah_visit_any, &x);
    occluded[i] = (uint8_t)x.accepted;
  }
}

typedef struct { ahp_record* out; uint32_t k, count; } ah_list_ctx;

static void ah_visit_list(void* vctx, const ahp_record* c)
{
  ah_list_ctx* x = (ah_list_ctx*)vctx;
  if (x->count < x->k) x->out[x->count] = *c;
  x->count++;
}

void ah_candidates(const orc_scene* s, const uint8_t* masks, const orc_ray* rays, uint64_t n, const uint32_t* rayMasks, const uint32_t* rayFlags,
                   uint32_t k, ahp_record* out, uint32_t* counts)
{
  for (uint64_t i = 0; i < n; ++i)
  {
    ah_list_ctx x = { out + i * (uint64_t)k, k, 0u };
    ah_each_candidate(s, masks, rayMasks[i], rayFlags[i], rays + i, ah_visit_list, &x);
    counts[i] = x.count;
  }
}
