// trace.cuh -- stack-based traversal of the two-level wide BVH and the watertight ray/triangle test.
//
// Replaces optixTrace (apps/rtigo3/shaders/raygeneration.cu:84-89 radiance rays, closesthit.cu:281-286
// shadow rays) and __anyhit__shadow (anyhit.cu:84-91).  B200 has no RT cores: boxes and triangles are
// tested on the FP32/INT pipes, nodes and triangles are fetched with 128-bit loads.
//
// The ARITHMETIC of the triangle test, of the object-space ray and of the hit ordering is a definition
// shared with the scalar oracle (oracle/rt_oracle.c "The ray/triangle test"); it is written with
// explicit round-to-nearest intrinsics so that the compiler's FMA contraction cannot change it.
// The box test is only required to be conservative and is free to use contracted arithmetic.
#pragma once

#include "rtc_internal.h"

#ifndef RTC_I2F_AXES
#define RTC_I2F_AXES 1            // number of axes (0, 1 or 2; swept with tools/sweep_i2f.sh: 1 and 2 are +0.4 %) whose plane bytes are converted by I2F.U8 instead of PRMT
#endif
#ifndef RTC_RESTORE_WORLD
#define RTC_RESTORE_WORLD 1       // world-space box constants restored from shared memory when an instance is left
#endif
#ifndef RTC_TRI_MINMAX
#define RTC_TRI_MINMAX 1          // mixed-sign test of the edge functions through FMNMX3 (see tri_test)
#endif
#ifndef RTC_LEAF_THRESHOLD
#define RTC_LEAF_THRESHOLD 0      // > 0: hold lanes with a pending leaf group back until this many lanes of the warp have one (trace_stream)
#endif
#ifndef RTC_ONE_TRI_PER_STEP
#define RTC_ONE_TRI_PER_STEP 0    // default of the TRICAP template parameter of Traversal / trace_stream (the kernels instantiate 0, 1 and 2 and pick per launch)
#endif
#ifndef RTC_FETCH_THRESHOLD
#define RTC_FETCH_THRESHOLD 12    // refill a warp when at least this many lanes have finished their ray (8: -1.3 %, 16: same; re-swept in round 2)
#endif
#ifndef RTC_TRACE_MIN_BLOCKS
#define RTC_TRACE_MIN_BLOCKS 8    // resident CTAs per SM the persistent traversal kernels are compiled for (register budget) and launched with
#endif

struct TraceHit
{
  float    t, u, v;
  uint32_t inst, prim;
};

// Shear constants of the current object-space ray (its origin is BoxRay::ox/oy/oz: inside an instance the box test and the
// triangle test share it).
struct ObjRay
{
  float dx, dy, dz;          // only live during the set-up at instance entry
  float Sx, Sy, Sz;
  int   kx, ky, kz;
};

// component k of (x, y, z) as two selects (a nested ternary compiles to divergent branches here)
__device__ __forceinline__ float sel3(float x, float y, float z, int k)
{
#if defined(__CUDACC__)
  float r;
  asm("{\n\t.reg .pred p1, p2;\n\tsetp.eq.s32 p1, %4, 1;\n\tsetp.eq.s32 p2, %4, 2;\n\tselp.f32 %0, %2, %1, p1;\n\tselp.f32 %0, %3, %0, p2;\n\t}"
      : "=&f"(r) : "f"(x), "f"(y), "f"(z), "r"(k));
  return r;
#else      // host build of this header (tests/native/trace_host.cpp): the same selection in C++
  return (k == 2) ? z : ((k == 1) ? y : x);
#endif
}

__device__ __forceinline__ void shear_setup(ObjRay& r)
{
  const float ax = fabsf(r.dx), ay = fabsf(r.dy), az = fabsf(r.dz);
  int kz = (ax >= ay && ax >= az) ? 0 : ((ay >= az) ? 1 : 2);
  int kx = kz + 1; if (kx == 3) kx = 0;
  int ky = kx + 1; if (ky == 3) ky = 0;
  const float dz = sel3(r.dx, r.dy, r.dz, kz);
  if (dz < 0.0f) { const int t = kx; kx = ky; ky = t; }
  r.kx = kx; r.ky = ky; r.kz = kz;
  r.Sx = __fdiv_rn(sel3(r.dx, r.dy, r.dz, kx), dz);
  r.Sy = __fdiv_rn(sel3(r.dx, r.dy, r.dz, ky), dz);
  r.Sz = __fdiv_rn(1.0f, dz);
}

// Woop/Benthin/Wald watertight test; see the oracle for the definition this mirrors operation by operation.
// The six component selections share their predicates (kx/ky/kz are per-ray constants): FSEL on three predicate pairs
// instead of a SETP pair in front of every select.
__device__ __forceinline__ float pick3(float x, float y, float z, bool is1, bool is2)
{
  float r = is1 ? y : x;
  return is2 ? z : r;
}

__device__ __forceinline__ bool tri_test(const ObjRay& r, float ox, float oy, float oz, const float4 v0, const float4 v1, const float4 v2,
                                         float& t, float& det, float& V, float& W)
{
  const float A0 = __fsub_rn(v0.x, ox), A1 = __fsub_rn(v0.y, oy), A2 = __fsub_rn(v0.z, oz);
  const float B0 = __fsub_rn(v1.x, ox), B1 = __fsub_rn(v1.y, oy), B2 = __fsub_rn(v1.z, oz);
  const float C0 = __fsub_rn(v2.x, ox), C1 = __fsub_rn(v2.y, oy), C2 = __fsub_rn(v2.z, oz);
  const bool x1 = r.kx == 1, x2 = r.kx == 2, y1 = r.ky == 1, y2 = r.ky == 2, z1 = r.kz == 1, z2 = r.kz == 2;
  const float Akz = pick3(A0, A1, A2, z1, z2), Bkz = pick3(B0, B1, B2, z1, z2), Ckz = pick3(C0, C1, C2, z1, z2);
  const float Ax = __fmaf_rn(-r.Sx, Akz, pick3(A0, A1, A2, x1, x2)), Ay = __fmaf_rn(-r.Sy, Akz, pick3(A0, A1, A2, y1, y2));
  const float Bx = __fmaf_rn(-r.Sx, Bkz, pick3(B0, B1, B2, x1, x2)), By = __fmaf_rn(-r.Sy, Bkz, pick3(B0, B1, B2, y1, y2));
  const float Cx = __fmaf_rn(-r.Sx, Ckz, pick3(C0, C1, C2, x1, x2)), Cy = __fmaf_rn(-r.Sy, Ckz, pick3(C0, C1, C2, y1, y2));
  float U = __fsub_rn(__fmul_rn(Cx, By), __fmul_rn(Cy, Bx));
  V = __fsub_rn(__fmul_rn(Ax, Cy), __fmul_rn(Ay, Cx));
  W = __fsub_rn(__fmul_rn(Bx, Ay), __fmul_rn(By, Ax));
  if (U == 0.0f || V == 0.0f || W == 0.0f)
  {
    U = (float)__dsub_rn(__dmul_rn((double)Cx, (double)By), __dmul_rn((double)Cy, (double)Bx));
    V = (float)__dsub_rn(__dmul_rn((double)Ax, (double)Cy), __dmul_rn((double)Ay, (double)Cx));
    W = (float)__dsub_rn(__dmul_rn((double)Bx, (double)Ay), __dmul_rn((double)By, (double)Ax));
  }
#if RTC_TRI_MINMAX
  // "one edge function negative and one positive" as min < 0 < max: two 3-input min/max and two compares instead of six
  // compares (identical for all non-NaN inputs; NaN edge functions need coordinates beyond 1e19)
  if (fminf(fminf(U, V), W) < 0.0f && fmaxf(fmaxf(U, V), W) > 0.0f) return false;
#else
  if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
#endif
  det = __fadd_rn(__fadd_rn(U, V), W);
  if (det == 0.0f) return false;
  const float Az = __fmul_rn(r.Sz, Akz), Bz = __fmul_rn(r.Sz, Bkz), Cz = __fmul_rn(r.Sz, Ckz);
  const float T = __fmaf_rn(U, Az, __fmaf_rn(V, Bz, __fmul_rn(W, Cz)));
  t = __fdiv_rn(T, det);
  return true;
}

// Per-space constants of the box test.
struct BoxRay
{
  float idx, idy, idz;       // 1/d (approximate reciprocal; the box test only has to be conservative), |d| clamped to 2^-80
  float ox, oy, oz;          // origin
  uint32_t octinv;           // 7 ^ octant, octant bit2 = dx<0, bit1 = dy<0, bit0 = dz<0
};

// EXACT = false: rcp.approx (the timed kernels; the box test only has to be conservative and its 2^-17 padding covers the
// approximation).  EXACT = true: IEEE reciprocal -- the counting kernels, whose node / triangle / instance counters the scalar
// oracle reproduces ray by ray on the exported BVH (oracle/wide_bvh.inc); rcp.approx has no portable definition.
template <bool EXACT>
__device__ __forceinline__ float fast_rcp(float d)
{
  if (fabsf(d) < 0x1p-80f) d = copysignf(0x1p-80f, d);
  if (EXACT) return __frcp_rn(d);
#if defined(__CUDACC__)
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
  return r;
#else      // host build: rcp.approx has no portable definition; the host harness only instantiates EXACT = true
  return 1.0f / d;
#endif
}

template <bool EXACT = false>
__device__ __forceinline__ void box_setup(BoxRay& b, float ox, float oy, float oz, float dx, float dy, float dz)
{
  b.idx = fast_rcp<EXACT>(dx); b.idy = fast_rcp<EXACT>(dy); b.idz = fast_rcp<EXACT>(dz);
  b.ox = ox; b.oy = oy; b.oz = oz;
  const uint32_t oct = ((dx < 0.0f) ? 4u : 0u) | ((dy < 0.0f) ? 2u : 0u) | ((dz < 0.0f) ? 1u : 0u);
  b.octinv = 7u ^ oct;
}

// 32768 + q as a float, q = byte i of w: one PRMT drops the byte into mantissa bits 8..15 of 0x47000000 (= 32768.0f),
// which replaces the shift/mask/I2F triple of a plain conversion.  The plane parameter is then ONE fma:
//   t = (32768 + q) * adj + (org - 32768 * adj),   adj = gridStep / d,  org = (p - o) / d.
// The cancellation costs at most 2^-9 grid steps, an eighth of the 1/64 step slack the builder guarantees.
// `bias` must hold 0x47000000 in a REGISTER (see node_test): with the constant as an immediate ptxas moves the byte selector
// into a fresh register before every PRMT, which doubles the cost of the decode.
template <uint32_t I>
__device__ __forceinline__ float quant_f(uint32_t w, uint32_t bias)
{
#if defined(__CUDACC__)
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(bias), "n"(0x7404u | (I << 4)));
  return __uint_as_float(r);
#else      // host build: selector 0x74I4 = {bias byte 3, bias byte 0, w byte I, bias byte 0} from the top byte down
  return __uint_as_float((bias & 0xff000000u) | ((bias & 0xffu) << 16) | (((w >> (8u * I)) & 0xffu) << 8) | (bias & 0xffu));
#endif
}

// q as a float through the conversion unit: one I2F.U8 with a byte selector.  It runs on the XU pipe, which the traversal
// barely uses, while PRMT competes with the selects, min/max and integer work for the ALU pipe (72 % busy on primary rays):
// RTC_I2F_AXES of the three axes are decoded this way to balance the two pipes.
template <uint32_t I>
__device__ __forceinline__ float quant_i2f(uint32_t w)
{
  return (float)((w >> (8u * I)) & 0xffu);
}

// 1/d of one axis saturated at 2^112 / gridStep (eb = the biased exponent of the grid step), so that |adj| <= 2^112 and the
// bias term 32768 * adj stays finite.  Saturation scales that axis's plane distances t by one factor s < 1, which keeps the
// near plane conservative; the far plane of a hit child keeps at least step / 64 of slack, so its scaled t stays >= 2^106,
// above every tmax < 2^100 (DESIGN.md section 3).  Unsaturated (grid steps up to 2^32 for any ray) the bits are unchanged.
// A plane origin term (p - o) / d that still overflows means the whole node lies more than 2^16 steps to one side of the
// origin, and the resulting +-inf culls exactly the boxes that lie entirely behind the origin or beyond tmax.
__device__ __forceinline__ float sat_idir(float id, uint32_t eb)
{
  const uint32_t raw = 0xB7000000u - (eb << 23);      // bits of 2^(112 - e) = 2^(239 - eb)
  const float lim = __uint_as_float(raw < 0x7F000000u ? raw : 0x7F000000u);   // at most 2^127
  return fminf(fmaxf(id, -lim), lim);
}

// Tests the 8 quantised child boxes of one node.  Returns bit s set when the box in slot s is hit.
// opaqueZero: a value that is always 0 but that the compiler cannot prove to be (bit 31 of a child index).
__device__ __forceinline__ uint32_t node_test(const BoxRay& b, const uint4 n0, const uint4 n2, const uint4 n3, const uint4 n4,
                                              float tmin, float tlimit, uint32_t opaqueZero)
{
  const uint32_t e = n0.w;
  const float idx = sat_idir(b.idx, e & 0xffu), idy = sat_idir(b.idy, (e >> 8) & 0xffu), idz = sat_idir(b.idz, (e >> 16) & 0xffu);
  const float adjx = __uint_as_float((e & 0xffu) << 23) * idx;
  const float adjy = __uint_as_float(((e >> 8) & 0xffu) << 23) * idy;
  const float adjz = __uint_as_float(((e >> 16) & 0xffu) << 23) * idz;
  const float orgx = fmaf(-32768.0f, adjx, (__uint_as_float(n0.x) - b.ox) * idx);
#if RTC_I2F_AXES >= 2
  const float orgy = (__uint_as_float(n0.y) - b.oy) * idy;
#else
  const float orgy = fmaf(-32768.0f, adjy, (__uint_as_float(n0.y) - b.oy) * idy);
#endif
#if RTC_I2F_AXES >= 1
  const float orgz = (__uint_as_float(n0.z) - b.oz) * idz;              // z planes: plain q through I2F, no bias to cancel
#else
  const float orgz = fmaf(-32768.0f, adjz, (__uint_as_float(n0.z) - b.oz) * idz);
#endif
  // near/far plane words per axis, selected by the direction sign
  // layout: n2 = qlox[0..3], qlox[4..7], qloy[0..3], qloy[4..7]; n3 = qloz, qhix; n4 = qhiy, qhiz
  const bool nx = b.idx < 0.0f, ny = b.idy < 0.0f, nz = b.idz < 0.0f;
  const uint32_t nearx[2] = { nx ? n3.z : n2.x, nx ? n3.w : n2.y }, farx[2] = { nx ? n2.x : n3.z, nx ? n2.y : n3.w };
  const uint32_t neary[2] = { ny ? n4.x : n2.z, ny ? n4.y : n2.w }, fary[2] = { ny ? n2.z : n4.x, ny ? n2.w : n4.y };
  const uint32_t nearz[2] = { nz ? n4.z : n3.x, nz ? n4.w : n3.y }, farz[2] = { nz ? n3.x : n4.z, nz ? n3.y : n4.w };
  const float tlimitPad = tlimit * (1.0f + 0x1p-17f);
  const uint32_t bias = 0x47000000u + opaqueZero;     // kept in a register on purpose, see quant_f
  uint32_t hits = 0;
#if RTC_I2F_AXES >= 1
#define RTC_QZ(I, W) quant_i2f<I>(W)
#else
#define RTC_QZ(I, W) quant_f<I>(W, bias)
#endif
#if RTC_I2F_AXES >= 2
#define RTC_QY(I, W) quant_i2f<I>(W)
#else
#define RTC_QY(I, W) quant_f<I>(W, bias)
#endif
#define RTC_BOX(S, H, I) \
  { \
    const float t0x = fmaf(quant_f<I>(nearx[H], bias), adjx, orgx), t1x = fmaf(quant_f<I>(farx[H], bias), adjx, orgx); \
    const float t0y = fmaf(RTC_QY(I, neary[H]), adjy, orgy), t1y = fmaf(RTC_QY(I, fary[H]), adjy, orgy); \
    const float t0z = fmaf(RTC_QZ(I, nearz[H]), adjz, orgz), t1z = fmaf(RTC_QZ(I, farz[H]), adjz, orgz); \
    const float tn = fmaxf(fmaxf(fmaxf(t0x, t0y), t0z), tmin); \
    const float tf = fminf(fminf(fminf(t1x, t1y), t1z) * (1.0f + 0x1p-17f), tlimitPad); \
    if (tn <= tf) hits |= 1u << S; \
  }
  RTC_BOX(0, 0, 0) RTC_BOX(1, 0, 1) RTC_BOX(2, 0, 2) RTC_BOX(3, 0, 3)
  RTC_BOX(4, 1, 0) RTC_BOX(5, 1, 1) RTC_BOX(6, 1, 2) RTC_BOX(7, 1, 3)
#undef RTC_BOX
#undef RTC_QZ
#undef RTC_QY
  return hits;
}

// bit s of an 8-bit mask -> bit (s ^ x)
__device__ __forceinline__ uint32_t xor_permute8(uint32_t h, uint32_t x)
{
  if (x & 1u) h = ((h & 0xAAu) >> 1) | ((h & 0x55u) << 1);
  if (x & 2u) h = ((h & 0xCCu) >> 2) | ((h & 0x33u) << 2);
  if (x & 4u) h = ((h & 0xF0u) >> 4) | ((h & 0x0Fu) << 4);
  return h;
}

// Per-ray work counters of the counting variant (the algorithmic-bytes figure of DESIGN.md section 5).
struct TraceCounts { uint32_t nodes, tris, insts; };

#define RTC_SM_STACK 8        // traversal stack entries per thread kept in shared memory
#if RTC_RESTORE_WORLD
#define RTC_SM_RAY_WORDS 15   // float columns per thread behind the stack (Traversal::smRay)
#else
#define RTC_SM_RAY_WORDS 11
#endif
#define RTC_LM_STACK 32       // overflow entries in local memory (never reached by the in-scope scenes)

// Rays whose traversal stack ran out of its 40 entries (the dropped subtree may hide a hit).  Never non-zero for the 8-wide
// trees this library builds; exported through rtc_stats so that a violation is loud instead of a silently wrong image.
// (one counter per translation unit that instantiates the traversal: kernels_trace.cu and kernels_shade.cu)
#ifndef RTC_STACK_OVERFLOW_COUNTER
#define RTC_STACK_OVERFLOW_COUNTER g_rtcStackOverflows
#endif
__device__ unsigned int RTC_STACK_OVERFLOW_COUNTER = 0;

// One ray's traversal as a resumable state machine: begin() once, then step() until it returns false.
// A step visits one wide node (or pops a postponed leaf group) and tests the triangles / enters the instance it yields.
// Closest hit (ANY = false): smallest t in (tmin, tmax), ties -> smaller (instance, primitive).  ANY = true: first hit ends the ray.
// SKIP = true (ordered any-hit processing of cutout materials, anyhit.cu:46-132): only candidates that come AFTER the key
// (skipT, skipInst, skipPrim) in the canonical order (t, instance, primitive) count, so repeated closest-hit queries
// enumerate the candidates of a ray in that order.
// TRICAP > 0 (rtc_context::traceSchedule, RTC_SCHEDULE_ONE_TRI / RTC_SCHEDULE_TWO_TRI): a step tests at most TRICAP triangles and a
// lane with more pending skips its node visit until they are done; see step().  0: every triangle of the leaves a node visit found.
template <bool ANY, bool COUNT, int BLOCK, bool SKIP = false, int TRICAP = RTC_ONE_TRI_PER_STEP>
struct Traversal
{
  float skipT; uint32_t skipInst, skipPrim;       // SKIP only
  // World ray origin/direction (needed only when an instance is entered or left) and the barycentric numerators of the
  // best hit (written once per accepted hit) live in shared memory, column-major like the stack: nine registers less,
  // which is what lets more CTAs fit on the SM.  Slots: 0-2 origin, 3-5 direction, 6 V, 7 W, 8 det, 9-10 triangle array of the
  // current GAS (pointer bits), 11-13 world 1/d and 14 the world octant word (restored when an instance is left instead of
  // recomputing three reciprocals).
  float* smRay;               // this thread's column: slot k at smRay[k * BLOCK]
  float tmin, tlimit;
  float hitT;                 // best t so far (the barycentric divisions are postponed to result(): same operands, same bits)
  uint32_t hitInst, hitPrim;
  // traversal state
  uint2 nodeGroup, triGroup;
  int sp, blasBase;
  uint32_t curInst;
  BoxRay br;
  ObjRay orr;
  const uint4*  nodes;
  uint2* smStack;             // this thread's column of the shared stack: entry k at smStack[k * BLOCK]
  uint2* lmStack;             // overflow entries (a local array owned by the caller)
  TraceCounts counts;

  __device__ __forceinline__ void push(uint2 v)
  {
    if (sp < RTC_SM_STACK) smStack[sp * BLOCK] = v;
    else if (sp < RTC_SM_STACK + RTC_LM_STACK) lmStack[sp - RTC_SM_STACK] = v;
    else { atomicAdd(&RTC_STACK_OVERFLOW_COUNTER, 1u); return; }
    ++sp;
  }
  __device__ __forceinline__ uint2 pop()
  {
    --sp;
    return (sp < RTC_SM_STACK) ? smStack[sp * BLOCK] : lmStack[(sp - RTC_SM_STACK) & (RTC_LM_STACK - 1)];
  }

  __device__ __forceinline__ bool found() const { return hitInst != 0xffffffffu; }

  __device__ __forceinline__ TraceHit result() const
  {
    TraceHit h;
    h.t = -1.0f; h.u = 0.0f; h.v = 0.0f; h.inst = 0xffffffffu; h.prim = 0xffffffffu;
    if (found())
    {
      h.t = hitT; h.inst = hitInst; h.prim = hitPrim;
      if (!ANY) { const float det = smRay[8 * BLOCK]; h.u = __fdiv_rn(smRay[6 * BLOCK], det); h.v = __fdiv_rn(smRay[7 * BLOCK], det); }
    }
    return h;
  }

  // returns false when the ray interval is empty (nothing to traverse)
  __device__ __forceinline__ bool begin(const SceneDesc& sc, const float4 o, const float4 d)
  {
    smRay[0] = o.x; smRay[BLOCK] = o.y; smRay[2 * BLOCK] = o.z;
    smRay[3 * BLOCK] = d.x; smRay[4 * BLOCK] = d.y; smRay[5 * BLOCK] = d.z;
    tmin = o.w; tlimit = d.w;
    hitT = -1.0f; hitInst = 0xffffffffu; hitPrim = 0xffffffffu;
    if (COUNT) { counts.nodes = 0; counts.tris = 0; counts.insts = 0; }
    if (!(tlimit > tmin)) return false;
    sp = 0; blasBase = -1; curInst = 0;
    box_setup<COUNT>(br, o.x, o.y, o.z, d.x, d.y, d.z);
#if RTC_RESTORE_WORLD
    smRay[11 * BLOCK] = br.idx; smRay[12 * BLOCK] = br.idy; smRay[13 * BLOCK] = br.idz; smRay[14 * BLOCK] = __uint_as_float(br.octinv);
#endif
    nodes = sc.tlasNodes;
    nodeGroup = make_uint2(0u, 0x80000000u);
    triGroup = make_uint2(0u, 0u);
    return true;
  }

  // A step = node_phase (visit one wide node, or take a popped leaf group) + leaf_phase (test the triangles / enter the
  // instance the leaf group holds) + advance (pop the next group, leave the instance, or finish).  The driver may run the
  // three for all lanes in every iteration (step) or hold lanes with a pending leaf group back until enough of them have
  // one (trace_stream, RTC_LEAF_THRESHOLD).
  __device__ __forceinline__ bool has_leaves() const { return triGroup.y != 0u; }

  __device__ __forceinline__ void node_phase()
  {
    if (nodeGroup.y & 0xff000000u)
    {
      const uint32_t bit = 31u - (uint32_t)__clz((int)nodeGroup.y);
      nodeGroup.y &= ~(1u << bit);
      if (nodeGroup.y & 0xff000000u) push(nodeGroup);
      const uint32_t slot = (bit - 24u) ^ br.octinv;
      const uint32_t rel = (uint32_t)__popc(nodeGroup.y & 0xffu & ((1u << slot) - 1u));
      const uint4* np = nodes + (size_t)(nodeGroup.x + rel) * 5u;
      const uint4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3), n4 = __ldg(np + 4);
      if (COUNT) counts.nodes++;
      const uint32_t hits = node_test(br, n0, n2, n3, n4, tmin, tlimit, n1.x >> 31);
      const uint32_t imask = n0.w >> 24;
      nodeGroup = make_uint2(n1.x, (xor_permute8(hits & imask, br.octinv) << 24) | imask);
      // leaf children: meta = (count << 5) | first primitive (relative to triBase)
      uint32_t leaf = hits & ~imask, primMask = 0u;
      while (leaf)
      {
        const uint32_t s = (uint32_t)__ffs((int)leaf) - 1u;
        leaf &= leaf - 1u;
        const uint32_t meta = (((s < 4u) ? n1.z : n1.w) >> (8u * (s & 3u))) & 0xffu;
        primMask |= ((1u << (meta >> 5)) - 1u) << (meta & 31u);
      }
      triGroup = make_uint2(n1.y, primMask);
    }
    else
    {
      triGroup = nodeGroup;
      nodeGroup = make_uint2(0u, 0u);
    }
  }

  // returns false when the ray is finished (ANY: first hit)
  __device__ __forceinline__ bool leaf_phase(const SceneDesc& sc)
  {
    int tested = 0;      // TRICAP > 1 only
    while (triGroup.y)
    {
      const uint32_t idx = (uint32_t)__ffs((int)triGroup.y) - 1u;
      triGroup.y &= triGroup.y - 1u;
      if (blasBase < 0)
      {
        // instance-level leaf: enter the instance
        const uint32_t inst = __ldg(sc.tlasLeaves + triGroup.x + idx);
        if (triGroup.y) push(triGroup);
        if (nodeGroup.y & 0xff000000u) push(nodeGroup);
        const float4* ip = sc.instances + (size_t)inst * 4u;
        const float4 r0 = __ldg(ip), r1 = __ldg(ip + 1), r2 = __ldg(ip + 2), r3 = __ldg(ip + 3);
        if (COUNT) counts.insts++;
        const float wox = smRay[0], woy = smRay[BLOCK], woz = smRay[2 * BLOCK];
        const float wdx = smRay[3 * BLOCK], wdy = smRay[4 * BLOCK], wdz = smRay[5 * BLOCK];
        const float oox = __fmaf_rn(r0.x, wox, __fmaf_rn(r0.y, woy, __fmaf_rn(r0.z, woz, r0.w)));
        const float ooy = __fmaf_rn(r1.x, wox, __fmaf_rn(r1.y, woy, __fmaf_rn(r1.z, woz, r1.w)));
        const float ooz = __fmaf_rn(r2.x, wox, __fmaf_rn(r2.y, woy, __fmaf_rn(r2.z, woz, r2.w)));
        orr.dx = __fmaf_rn(r0.x, wdx, __fmaf_rn(r0.y, wdy, __fmul_rn(r0.z, wdz)));
        orr.dy = __fmaf_rn(r1.x, wdx, __fmaf_rn(r1.y, wdy, __fmul_rn(r1.z, wdz)));
        orr.dz = __fmaf_rn(r2.x, wdx, __fmaf_rn(r2.y, wdy, __fmul_rn(r2.z, wdz)));
        shear_setup(orr);
        box_setup<COUNT>(br, oox, ooy, ooz, orr.dx, orr.dy, orr.dz);
        curInst = inst;
        blasBase = sp;
        nodes = reinterpret_cast<const uint4*>(((unsigned long long)__float_as_uint(r3.y) << 32) | __float_as_uint(r3.x));
        smRay[9 * BLOCK] = r3.z; smRay[10 * BLOCK] = r3.w;
        nodeGroup = make_uint2(0u, 0x80000000u);
        triGroup = make_uint2(0u, 0u);
        break;
      }
      else
      {
        const float4* tris = reinterpret_cast<const float4*>(((unsigned long long)__float_as_uint(smRay[10 * BLOCK]) << 32) | __float_as_uint(smRay[9 * BLOCK]));
        const float4* tp = tris + (size_t)(triGroup.x + idx) * 3u;
        const float4 v0 = __ldg(tp), v1 = __ldg(tp + 1), v2 = __ldg(tp + 2);
        if (COUNT) counts.tris++;
        float t, det, V, W;
        if (tri_test(orr, br.ox, br.oy, br.oz, v0, v1, v2, t, det, V, W) && t > tmin)
        {
          const uint32_t prim = __float_as_uint(v0.w);
          if (SKIP && !(t > skipT || (t == skipT && (curInst > skipInst || (curInst == skipInst && prim > skipPrim))))) continue;
          if (ANY)
          {
            if (t < tlimit) { hitT = t; hitInst = curInst; hitPrim = prim; return false; }
          }
          else
          {
            const bool better = found() ? (t < hitT || (t == hitT && (curInst < hitInst || (curInst == hitInst && prim < hitPrim))))
                                      : (t < tlimit);
            if (better)
            {
              tlimit = t;
              hitT = t; hitInst = curInst; hitPrim = prim;
              smRay[6 * BLOCK] = V; smRay[7 * BLOCK] = W; smRay[8 * BLOCK] = det;
            }
          }
        }
        if (TRICAP == 1 || (TRICAP > 1 && ++tested >= TRICAP)) break;
      }
    }
    return true;
  }

  // returns false when the traversal is complete
  __device__ __forceinline__ bool advance(const SceneDesc& sc)
  {
    if (!(nodeGroup.y & 0xff000000u))
    {
      if (blasBase >= 0 && sp == blasBase)
      {
        blasBase = -1;   // leave the instance: back to the world-space ray
        nodes = sc.tlasNodes;
#if RTC_RESTORE_WORLD
        br.ox = smRay[0]; br.oy = smRay[BLOCK]; br.oz = smRay[2 * BLOCK];
        br.idx = smRay[11 * BLOCK]; br.idy = smRay[12 * BLOCK]; br.idz = smRay[13 * BLOCK]; br.octinv = __float_as_uint(smRay[14 * BLOCK]);
#else
        box_setup<COUNT>(br, smRay[0], smRay[BLOCK], smRay[2 * BLOCK], smRay[3 * BLOCK], smRay[4 * BLOCK], smRay[5 * BLOCK]);
#endif
      }
      if (sp == 0) return false;
      nodeGroup = pop();
    }
    return true;
  }

  // returns true while the ray needs more steps
  __device__ __forceinline__ bool step(const SceneDesc& sc)
  {
    if (TRICAP > 0)
    {
      // A warp pays the triangle loop of an iteration for as long as its unluckiest lane: 3.2 tests per iteration on bounce
      // rays of the geometry scene, although a lane tests 0.4 triangles per node visit on average.  Here a step tests at most
      // TRICAP triangles (one, or two = one leaf of the host builder), and a lane with more of them pending skips its node
      // visit, so an iteration costs one node pass plus TRICAP triangle passes.  Per ray nothing changes -- the same tests in
      // the same order, identical hits and work counters (tests/test_cpu_trace_source.py) -- only their timing within the
      // warp: with a cap of one 26 % more iterations and 60 % fewer triangle passes, with two 6 % and 40 % (tests/tools/simd_cost.py).
      // Built after the last GPU session of round 2 and therefore never enabled blindly: the library times one batch with each
      // schedule and keeps a capped one only where it is faster (kernels_shade.cu, "schedule tuner").
      if (!(blasBase >= 0 && has_leaves())) node_phase();
      if (!leaf_phase(sc)) return false;
      if (blasBase >= 0 && has_leaves()) return true;
      return advance(sc);
    }
    node_phase();
    if (!leaf_phase(sc)) return false;
    return advance(sc);
  }
};

// Persistent-warp driver: every lane owns one ray at a time; lanes whose ray has finished take the next ray index from a
// global cursor (one atomicAdd per warp and refill), so short rays do not leave their lanes idle while the longest ray of
// the warp finishes.  Policy (stateless) supplies load(i, org, dir, tag) -> bool (false: skip this
// index; tag = the policy's per-ray word, e.g. the path id), store(tag, hit) and, for SKIP kernels, skip_key(tag, t, inst, prim).
template <bool ANY, bool COUNT, int BLOCK, bool SKIP, int TRICAP = RTC_ONE_TRI_PER_STEP, class Policy>
__device__ __forceinline__ void trace_stream(const SceneDesc& sc, uint32_t n, uint32_t* __restrict__ cursor, Policy& policy, uint2* smem,
                                             unsigned long long* __restrict__ countsOut)
{
  Traversal<ANY, COUNT, BLOCK, SKIP, TRICAP> tr;
  uint2 overflow[RTC_LM_STACK];
  tr.smStack = smem + threadIdx.x;
  tr.smRay = reinterpret_cast<float*>(smem + RTC_SM_STACK * BLOCK) + threadIdx.x;
  tr.lmStack = overflow;
  const uint32_t lane = threadIdx.x & 31u;
  bool active = false, exhausted = false;
  uint32_t tag = 0;
  unsigned long long cNodes = 0, cTris = 0, cInsts = 0, cRays = 0;
  for (;;)
  {
    const uint32_t idle = __ballot_sync(0xffffffffu, !active);
    if (idle && !exhausted && (idle == 0xffffffffu || __popc(idle) >= RTC_FETCH_THRESHOLD))
    {
      const uint32_t want = (uint32_t)__popc(idle);
      const uint32_t leader = (uint32_t)__ffs((int)idle) - 1u;
      uint32_t base = 0;
      if (lane == leader) base = atomicAdd(cursor, want);
      base = __shfl_sync(0xffffffffu, base, leader);
      if (base + want >= n) exhausted = true;
      if (!active)
      {
        const uint32_t index = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
        if (index < n)
        {
          float4 o, d;
          if (policy.load(index, o, d, tag))
          {
            if constexpr (SKIP) policy.skip_key(tag, tr.skipT, tr.skipInst, tr.skipPrim);
            if (tr.begin(sc, o, d)) active = true;
            else { policy.store(tag, tr.result()); if (COUNT) cRays++; }
          }
        }
      }
    }
    else if (idle == 0xffffffffu) break;      // nothing running and nothing left to fetch
#if RTC_LEAF_THRESHOLD > 0
    // Lanes whose node visit produced a leaf group (triangles to test or an instance to enter) are HELD BACK -- they skip
    // node visits -- until RTC_LEAF_THRESHOLD lanes of the warp hold one (or a quarter of the running lanes, or nobody can
    // visit a node any more); then all of them run the leaf phase together.  Nothing is reordered inside a ray; the leaf
    // phase, which a warp used to run in almost every iteration for the ~3 lanes that had just found a leaf, runs every
    // second or third iteration for 8+ lanes instead.
    bool running = active;
    if (active && !tr.has_leaves()) tr.node_phase();
    const bool held = active && tr.has_leaves();
    const uint32_t heldLanes = __ballot_sync(0xffffffffu, held), activeLanes = ~idle;
    if (heldLanes)
    {
      const uint32_t nHeld = (uint32_t)__popc(heldLanes), nActive = (uint32_t)__popc(activeLanes);
      if (nHeld >= RTC_LEAF_THRESHOLD || nHeld * 4u >= nActive)
      {
        if (held) running = tr.leaf_phase(sc);
      }
    }
    if (running && !tr.has_leaves()) running = tr.advance(sc);
    if (active && !running)
    {
      policy.store(tag, tr.result());
      if (COUNT) { cNodes += tr.counts.nodes; cTris += tr.counts.tris; cInsts += tr.counts.insts; cRays++; }
      active = false;
    }
#else
    if (active)
    {
      if (!tr.step(sc))
      {
        policy.store(tag, tr.result());
        if (COUNT) { cNodes += tr.counts.nodes; cTris += tr.counts.tris; cInsts += tr.counts.insts; cRays++; }
        active = false;
      }
    }
#endif
  }
  if (COUNT)
  {
    for (int off = 16; off; off >>= 1)
    {
      cNodes += __shfl_down_sync(0xffffffffu, cNodes, off); cTris += __shfl_down_sync(0xffffffffu, cTris, off);
      cInsts += __shfl_down_sync(0xffffffffu, cInsts, off); cRays += __shfl_down_sync(0xffffffffu, cRays, off);
    }
    if (lane == 0 && cRays)
    {
      atomicAdd(countsOut + 0, cNodes); atomicAdd(countsOut + 1, cTris); atomicAdd(countsOut + 2, cInsts); atomicAdd(countsOut + 3, cRays);
    }
  }
}
