// primary_lists.cuh -- per-tile candidate lists of the primary rays of a pinhole launch (DESIGN.md section 3, "Tile lists").
//
// A warp of the depth-0 extend is one 8x4-pixel tile of one iteration, and a batch traces every tile once per iteration.  With
// the pinhole lens every primary ray of a tile starts at cam.P and points into the tile's pixel rectangle, so the triangles any
// of them can hit lie in the tile's frustum.  build_tile_list collects them once per tile and batch; trace_tile_list then runs
// the traversal's own triangle test (tri_test, enter_instance, closer_hit) over that list for each ray.  Closest hit is a total
// order on (t, instance, primitive), so any superset of the triangles the traversal can accept gives the traversal's bits.
//
// Conservativeness.  A side plane of the frustum goes through the apex P with outward unit normal n; a point v is OUTSIDE it
// when n.(v - P) > kFrustumPad |v - P|, i.e. more than asin(2^-12) beyond the plane as seen from P.  A triangle is dropped only
// when its three vertices are outside one plane, a box only when all of it is.  The padding has to cover every rounding between
// the exact frustum and what tri_test accepts, as an angle seen from the apex:
//   * the side normals (tile_planes): each is the cross product of two vectors at least asin(1/8) apart (U a + W and V, or U
//     and V b + W), never of two corner directions of the tile, which are nearly parallel and would lose precision as 2^-24
//     over the tile's angle; error a few 2^-24 times 8.  In object space the normal is cof(M) n with the cofactor matrix of the
//     world->object rows M, whose relative error is a few 2^-24 times the condition number |M|_F |M^-1|_F, held to
//     kMaxCondition = 64 (a tile that meets a worse instance is traced by the traversal instead).  Emulated in float32 over
//     random tiles (fields of view 60, 3 and 1 degrees, 1080p and 4K, an instance squashed to |M|_F |M^-1|_F = 57), the
//     farthest an exact boundary ray of a tile falls outside its computed plane is 0.0024 of the padding;
//   * the ndc bounds of the tile (approximate reciprocal of the resolution) and the ray generation (fragment, ndc, the
//     -fmad=false combination of U, V, W, normalize): a few 2^-24;
//   * enter_instance: the object-space apex is the very value tri_test takes (the builder makes the same call); the direction
//     rows add a few 2^-24 times the condition number;
//   * the shear and the edge functions of tri_test: a few 2^-24 each, relative to the vertices' distances from the origin;
//   * the builder's own square roots and reciprocals (MUFU approximations on the device): relative 2^-22.
// With the condition number at its limit of 64 that is below 2^-15 in all, an eighth of the padding.  The one case those
// relative bounds do not cover is a triangle whose plane passes (nearly) through the apex: seen edge-on, the rounded edge
// functions can agree in sign for rays that pass beside it.  Such a triangle is never dropped (the edge-on rule in
// tri_maybe_hit).  Child boxes are decoded from the quantised planes and rounded outward, so they contain whatever the
// traversal's boxes contain.
#pragma once

#include "trace.cuh"

#ifndef RTC_TILE_LIST_K
#define RTC_TILE_LIST_K 16        // entries per tile list (DESIGN.md section 3); a tile with more candidates is traced by the traversal
#endif
constexpr uint32_t kTileListK = RTC_TILE_LIST_K;
constexpr uint32_t kTileOverflow = 0xffffffffu;   // count of a tile whose candidates do not fit (or that meets an ill-conditioned instance)
constexpr float kFrustumPad = 0x1p-12f;
constexpr float kMaxCondition = 64.0f;
#define RTC_FRUSTUM_STACK 64      // pending nodes of one walk; deeper means overflow, never a dropped subtree

// Square root and reciprocal square root of the list builder: MUFU approximations on the device (relative error below 2^-22,
// far inside the padding; the IEEE versions this translation unit would otherwise compile are subroutine calls), IEEE on the host.
__device__ __forceinline__ float pl_rsqrt(float x)
{
#if defined(__CUDACC__)
  return rsqrtf(x);
#else
  return 1.0f / sqrtf(x);
#endif
}
__device__ __forceinline__ float pl_sqrt(float x) { return x * pl_rsqrt(fmaxf(x, 0x1p-126f)); }

// The four side planes of a tile's frustum in one space: apex and outward unit normals.
struct TileFrustum
{
  float px, py, pz;
  float nx[4], ny[4], nz[4];
};

// n[k]: normal of side plane k (any length), c: a direction inside the frustum.  The normals are normalised and turned outward.
__device__ __forceinline__ void make_frustum(TileFrustum& f, float px, float py, float pz, const float n[4][3], const float c[3])
{
  f.px = px; f.py = py; f.pz = pz;
  for (int k = 0; k < 4; ++k)
  {
    const float x = n[k][0], y = n[k][1], z = n[k][2];
    float s = pl_rsqrt(x * x + y * y + z * z);
    if (x * c[0] + y * c[1] + z * c[2] > 0.0f) s = -s;
    f.nx[k] = x * s; f.ny[k] = y * s; f.nz[k] = z * s;
  }
}

// bit k set: (x, y, z) is outside plane k.  NaN never counts as outside.
__device__ __forceinline__ uint32_t outside_mask(const TileFrustum& f, float x, float y, float z)
{
  const float dx = x - f.px, dy = y - f.py, dz = z - f.pz;
  const float pad = kFrustumPad * pl_sqrt(dx * dx + dy * dy + dz * dz);
  uint32_t m = 0;
  for (int k = 0; k < 4; ++k)
    if (f.nx[k] * dx + f.ny[k] * dy + f.nz[k] * dz > pad) m |= 1u << k;
  return m;
}

__device__ __forceinline__ bool box_outside(const TileFrustum& f, float lox, float loy, float loz, float hix, float hiy, float hiz)
{
  const float hx = 0.5f * (hix - lox), hy = 0.5f * (hiy - loy), hz = 0.5f * (hiz - loz);
  const float dx = 0.5f * (lox + hix) - f.px, dy = 0.5f * (loy + hiy) - f.py, dz = 0.5f * (loz + hiz) - f.pz;
  // every point v of the box has n.(v - P) >= n.(c - P) - sum |n_i| h_i and |v - P| <= |c - P| + |h|
  const float pad = kFrustumPad * (pl_sqrt(dx * dx + dy * dy + dz * dz) + pl_sqrt(hx * hx + hy * hy + hz * hz));
  for (int k = 0; k < 4; ++k)
  {
    const float near = f.nx[k] * dx + f.ny[k] * dy + f.nz[k] * dz - (fabsf(f.nx[k]) * hx + fabsf(f.ny[k]) * hy + fabsf(f.nz[k]) * hz);
    if (near > pad) return true;
  }
  return false;
}

// false only when no ray of the frustum can be accepted by tri_test on this triangle
__device__ __forceinline__ bool tri_maybe_hit(const TileFrustum& f, const float4 v0, const float4 v1, const float4 v2)
{
  if (outside_mask(f, v0.x, v0.y, v0.z) & outside_mask(f, v1.x, v1.y, v1.z) & outside_mask(f, v2.x, v2.y, v2.z))
  {
    // edge-on rule: keep the triangle when the apex lies within the padding angle of its plane (degenerate ones included)
    const float ax = v1.x - v0.x, ay = v1.y - v0.y, az = v1.z - v0.z, bx = v2.x - v0.x, by = v2.y - v0.y, bz = v2.z - v0.z;
    const float nx = ay * bz - az * by, ny = az * bx - ax * bz, nz = ax * by - ay * bx;
    const float dx = v0.x - f.px, dy = v0.y - f.py, dz = v0.z - f.pz;
    const float r0 = dx * dx + dy * dy + dz * dz;
    const float r1 = (v1.x - f.px) * (v1.x - f.px) + (v1.y - f.py) * (v1.y - f.py) + (v1.z - f.pz) * (v1.z - f.pz);
    const float r2 = (v2.x - f.px) * (v2.x - f.px) + (v2.y - f.py) * (v2.y - f.py) + (v2.z - f.pz) * (v2.z - f.pz);
    const float rmax = pl_sqrt(fmaxf(fmaxf(r0, r1), r2));
    return !(fabsf(nx * dx + ny * dy + nz * dz) > kFrustumPad * pl_sqrt(nx * nx + ny * ny + nz * nz) * rmax);
  }
  return true;
}

// Child s of a wide node as a float box, rounded outward (the quantised planes are exact multiples of the grid step).
__device__ __forceinline__ void child_box(const uint4 n0, const uint4 n2, const uint4 n3, const uint4 n4, uint32_t s, float lo[3], float hi[3])
{
  const uint32_t sh = 8u * (s & 3u);
  const bool h = s >= 4u;
  const uint32_t q[6] = { ((h ? n2.y : n2.x) >> sh) & 0xffu, ((h ? n2.w : n2.z) >> sh) & 0xffu, ((h ? n3.y : n3.x) >> sh) & 0xffu,
                          ((h ? n3.w : n3.z) >> sh) & 0xffu, ((h ? n4.y : n4.x) >> sh) & 0xffu, ((h ? n4.w : n4.z) >> sh) & 0xffu };
  const float p[3] = { __uint_as_float(n0.x), __uint_as_float(n0.y), __uint_as_float(n0.z) };
  for (int a = 0; a < 3; ++a)
  {
    const float step = __uint_as_float(((n0.w >> (8u * a)) & 0xffu) << 23);
    const float l = p[a] + (float)q[a] * step, u = p[a] + (float)q[3 + a] * step;
    lo[a] = l - fabsf(l) * 0x1p-22f; hi[a] = u + fabsf(u) * 0x1p-22f;
  }
}

// Depth-first walk of a wide BVH: leaf(primitive index) for every primitive of every leaf whose box is not outside the frustum.
// Returns false as soon as leaf() does or the stack runs out.
template <class Leaf>
__device__ __forceinline__ bool frustum_walk(const uint4* nodes, const TileFrustum& f, Leaf&& leaf)
{
  uint32_t stack[RTC_FRUSTUM_STACK];
  int sp = 0;
  uint32_t node = 0;
  for (;;)
  {
    const uint4* np = nodes + (size_t)node * 5u;
    const uint4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
    const uint32_t imask = n0.w >> 24;
    for (uint32_t s = 0; s < 8u; ++s)
    {
      const bool inner = (imask >> s) & 1u;
      const uint32_t meta = (((s < 4u) ? n1.z : n1.w) >> (8u * (s & 3u))) & 0xffu;
      if (!inner && meta == 0u) continue;
      float lo[3], hi[3];
      child_box(n0, n2, n3, n4, s, lo, hi);
      if (box_outside(f, lo[0], lo[1], lo[2], hi[0], hi[1], hi[2])) continue;
      if (inner)
      {
        if (sp == RTC_FRUSTUM_STACK) return false;
        stack[sp++] = n1.x + (uint32_t)__popc(imask & ((1u << s) - 1u));
      }
      else
      {
        for (uint32_t j = 0; j < (meta >> 5); ++j)
          if (!leaf(n1.y + (meta & 31u) + j)) return false;
      }
    }
    if (sp == 0) return true;
    node = stack[--sp];
  }
}

__device__ __forceinline__ void cross3(const float a[3], const float b[3], float r[3])
{
  r[0] = a[1] * b[2] - a[2] * b[1]; r[1] = a[2] * b[0] - a[0] * b[2]; r[2] = a[0] * b[1] - a[1] * b[0];
}

// World-space frustum of the tile whose top-left pixel is (x0, y0): apex cam.P, the normals of the four side planes and the
// tile's centre direction.  The pinhole directions of the tile are U a + V b + W for ndc a in [a0, a1], b in [b0, b1]
// (fragments x0 .. x0 + 8, y0 .. y0 + 4).  The plane at a = a0 is spanned by U a0 + W and V, the one at b = b0 by U and
// V b0 + W: each normal is the cross product of two vectors at a wide angle, so it keeps a relative error of a few 2^-24.  (The
// cross product of two corner directions of a tile, which are nearly parallel, would lose precision as 2^-24 over the tile's
// angle.)  Returns false when a pair is closer than asin(1/8) to parallel (a degenerate camera): the tile is not listed.
__device__ __forceinline__ bool tile_planes(const rt_SystemData& sys, uint32_t x0, uint32_t y0, float P[3], float n[4][3], float c[3])
{
  const rt_CameraDefinition& cam = reinterpret_cast<const rt_CameraDefinition*>(sys.cameraDefinitions)[0];
  const float isx = fast_rcp<false>((float)sys.resolution.x), isy = fast_rcp<false>((float)sys.resolution.y);
  const float a[2] = { ((float)x0 * isx) * 2.0f - 1.0f, ((float)(x0 + 8u) * isx) * 2.0f - 1.0f };
  const float b[2] = { ((float)y0 * isy) * 2.0f - 1.0f, ((float)(y0 + 4u) * isy) * 2.0f - 1.0f };
  const float U[3] = { cam.U.x, cam.U.y, cam.U.z }, V[3] = { cam.V.x, cam.V.y, cam.V.z }, W[3] = { cam.W.x, cam.W.y, cam.W.z };
  P[0] = cam.P.x; P[1] = cam.P.y; P[2] = cam.P.z;
  const float am = 0.5f * (a[0] + a[1]), bm = 0.5f * (b[0] + b[1]);
  for (int i = 0; i < 3; ++i) c[i] = U[i] * am + V[i] * bm + W[i];
  bool ok = true;
  for (int k = 0; k < 4; ++k)
  {
    float e[3], f[3];
    for (int i = 0; i < 3; ++i)
    {
      e[i] = (k < 2) ? U[i] * a[k] + W[i] : U[i];
      f[i] = (k < 2) ? V[i] : V[i] * b[k - 2] + W[i];
    }
    cross3(e, f, n[k]);
    const float nn = n[k][0] * n[k][0] + n[k][1] * n[k][1] + n[k][2] * n[k][2];
    const float ee = e[0] * e[0] + e[1] * e[1] + e[2] * e[2], ff = f[0] * f[0] + f[1] * f[1] + f[2] * f[2];
    ok = ok && nn * 64.0f >= ee * ff;
  }
  return ok;
}

// The candidate list of one tile: rays from P into the frustum of tile_planes (side normals n, centre direction c).  Writes
// (instance, triangle record index) pairs grouped by instance to out[0 .. K) and returns their number, or kTileOverflow.
__device__ __forceinline__ uint32_t build_tile_list(const SceneDesc& sc, const float P[3], const float n[4][3], const float c[3], uint2* out)
{
  TileFrustum wf;
  make_frustum(wf, P[0], P[1], P[2], n, c);
  uint32_t count = 0;
  const bool ok = frustum_walk(sc.tlasNodes, wf, [&](uint32_t leafIndex) -> bool {
    const uint32_t inst = __ldg(sc.tlasLeaves + leafIndex);
    const float4* ip = sc.instances + (size_t)inst * 4u;
    const float4 r0 = __ldg(ip), r1 = __ldg(ip + 1), r2 = __ldg(ip + 2), r3 = __ldg(ip + 3);
    // object space: the rows M map directions, the cofactor matrix cof(M) = det(M) M^-T maps plane normals
    const float m[3][3] = { { r0.x, r0.y, r0.z }, { r1.x, r1.y, r1.z }, { r2.x, r2.y, r2.z } };
    float cof[3][3];
    cross3(m[1], m[2], cof[0]); cross3(m[2], m[0], cof[1]); cross3(m[0], m[1], cof[2]);
    const float det = m[0][0] * cof[0][0] + m[0][1] * cof[0][1] + m[0][2] * cof[0][2];
    float fm = 0.0f, fc = 0.0f;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) { fm += m[i][j] * m[i][j]; fc += cof[i][j] * cof[i][j]; }
    if (!(fm * fc <= kMaxCondition * kMaxCondition * det * det)) return false;     // |M|_F |M^-1|_F > kMaxCondition (or NaN)
    // the object-space apex with the bits tri_test will see
    ObjRay orr; float ox, oy, oz;
    enter_instance(r0, r1, r2, P[0], P[1], P[2], c[0], c[1], c[2], orr, ox, oy, oz);
    float on[4][3], oc[3];
    for (int i = 0; i < 3; ++i)
    {
      oc[i] = m[i][0] * c[0] + m[i][1] * c[1] + m[i][2] * c[2];
      for (int k = 0; k < 4; ++k) on[k][i] = cof[i][0] * n[k][0] + cof[i][1] * n[k][1] + cof[i][2] * n[k][2];
    }
    TileFrustum of;
    make_frustum(of, ox, oy, oz, on, oc);
    const uint4* nodes = reinterpret_cast<const uint4*>(((unsigned long long)__float_as_uint(r3.y) << 32) | __float_as_uint(r3.x));
    const float4* tris = reinterpret_cast<const float4*>(((unsigned long long)__float_as_uint(r3.w) << 32) | __float_as_uint(r3.z));
    return frustum_walk(nodes, of, [&](uint32_t tri) -> bool {
      const float4* tp = tris + (size_t)tri * 3u;
      if (!tri_maybe_hit(of, __ldg(tp), __ldg(tp + 1), __ldg(tp + 2))) return true;
      if (count == kTileListK) return false;
      out[count++] = make_uint2(inst, tri);
      return true;
    });
  });
  return ok ? count : kTileOverflow;
}

// Closest hit of one ray (o.xyz, tmin) (d.xyz, tmax) over a tile's list, with exactly the traversal's arithmetic: enter_instance
// at each change of instance, tri_test, t > tmin and closer_hit per entry, the barycentric divisions of Traversal::result.
// The list is read by all lanes of a warp at once.
__device__ __forceinline__ TraceHit trace_tile_list(const SceneDesc& sc, const uint2* list, uint32_t count, const float4 o, const float4 d)
{
  TraceHit h;
  h.t = -1.0f; h.u = 0.0f; h.v = 0.0f; h.inst = 0xffffffffu; h.prim = 0xffffffffu;
  if (!(d.w > o.w)) return h;                  // Traversal::begin: empty interval
  float hitT = -1.0f, bestV = 0.0f, bestW = 0.0f, bestDet = 1.0f;
  uint32_t hitInst = 0xffffffffu, hitPrim = 0xffffffffu, cur = 0xffffffffu;
  ObjRay orr; float ox = 0.0f, oy = 0.0f, oz = 0.0f;
  const float4* tris = nullptr;
  for (uint32_t e = 0; e < count; ++e)
  {
    const uint2 en = __ldg(list + e);
    if (en.x != cur)
    {
      const float4* ip = sc.instances + (size_t)en.x * 4u;
      const float4 r0 = __ldg(ip), r1 = __ldg(ip + 1), r2 = __ldg(ip + 2), r3 = __ldg(ip + 3);
      enter_instance(r0, r1, r2, o.x, o.y, o.z, d.x, d.y, d.z, orr, ox, oy, oz);
      tris = reinterpret_cast<const float4*>(((unsigned long long)__float_as_uint(r3.w) << 32) | __float_as_uint(r3.z));
      cur = en.x;
    }
    const float4* tp = tris + (size_t)en.y * 3u;
    const float4 v0 = __ldg(tp), v1 = __ldg(tp + 1), v2 = __ldg(tp + 2);
    float t, det, V, W;
    if (tri_test(orr, ox, oy, oz, v0, v1, v2, t, det, V, W) && t > o.w)
    {
      const uint32_t prim = __float_as_uint(v0.w);
      if (closer_hit(t, cur, prim, hitT, hitInst, hitPrim, d.w))
      {
        hitT = t; hitInst = cur; hitPrim = prim; bestV = V; bestW = W; bestDet = det;
      }
    }
  }
  if (hitInst != 0xffffffffu)
  {
    h.t = hitT; h.inst = hitInst; h.prim = hitPrim;
    h.u = __fdiv_rn(bestV, bestDet); h.v = __fdiv_rn(bestW, bestDet);
  }
  return h;
}
