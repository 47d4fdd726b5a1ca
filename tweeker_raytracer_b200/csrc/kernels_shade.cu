// kernels_shade.cu -- the shading side of the wavefront integrator: generate, shade, accumulate, plus
// composite, tonemap and primary-ray export.  Built with -fmad=false (see shade.cuh).
//
//   generate   = __raygen__path_tracer prologue          (raygeneration.cu:173-201, :44-59)
//   shade      = __closesthit__radiance / __miss__env_*  (closesthit.cu:126-279, miss.cu:41-109)
//                + the integrator epilogue               (raygeneration.cu:92-145)
//   accumulate = NaN filter + running average            (raygeneration.cu:220-253, :312-342)
//   composite  = compositor kernel                       (compositor.cu:38-65)
//   tonemap    = Application::screenshot loop            (Application.cpp:2262-2295)
//
// Path state lives in SoA arrays indexed by path id (WavefrontBuffers); queues hold path ids and are
// compacted with warp ballots (one atomicAdd per warp).
#include "shade.cuh"
// the primary-ray extend kernel generates its rays with the shading arithmetic of this translation unit (see ExtendPrimary)
#define RTC_STACK_OVERFLOW_COUNTER g_rtcStackOverflowsPrimary
#include "trace.cuh"
#include "schedule_tuner.h"

#include <cstdlib>
#include <cstring>

namespace {

constexpr int kBlock = 256;
constexpr uint32_t kNoPixel = 0xffffffffu;
constexpr uint32_t kDeadPath = 0xfffffffeu;           // hitInst of a launch index that falls outside the image (fused primary path)
// device counters of one batch: [0..63] extend counts per depth, [64..127] shadow counts, [128..191] extend cursors,
// [192..255] connect cursors, [256 + 8 d + c] paths of shade class c at depth d
constexpr uint32_t kNumCounters = 256 + 64 * 8;
constexpr uint32_t kPendingRR = 0x80000000u;          // misc.y bit: Russian roulette postponed until the shadow ray is resolved
constexpr uint32_t kDepthMask = 0x0000ffffu;
constexpr uint64_t kMaxPathsInFlight = 64ull << 20;   // 64 Mi paths x 320 B of wavefront state = 21 GB of the 180 GB HBM

struct WfArgs
{
  WavefrontBuffers wf;
  rt_SystemData sys;
  uint32_t launchWidth, launchHeight;
  int raygen, miss;
  int iterFirst, iterCount;
  int accumFirst;          // sample number of the batch's first iteration in the running average
  uint32_t numPaths;
};

// Launch-index order of the wavefront: consecutive path ids cover 8x4 pixel tiles (a warp = one tile) instead of 32x1
// row segments, which keeps the rays of a warp closer together.  Falls back to row-major when the launch does not tile.
__device__ __forceinline__ void launch_xy(uint32_t idx, uint32_t w, uint32_t h, uint32_t& x, uint32_t& y)
{
  if (((w & 7u) | (h & 3u)) == 0u)
  {
    const uint32_t tile = idx >> 5, within = idx & 31u, tilesPerRow = w >> 3;
    const uint32_t ty = tile / tilesPerRow, tx = tile - ty * tilesPerRow;
    x = (tx << 3) + (within & 7u);
    y = (ty << 2) + (within >> 3);
  }
  else
  {
    y = idx / w; x = idx - y * w;
  }
}

// Queue append aggregated over the whole CTA: every thread offers (class, value), class < 0 meaning nothing.  Lanes of a
// warp with the same class are found with one ballot per class (NCLS is small; match.any is several times slower), each
// warp reserves its run in a shared counter, ONE thread per class reserves the CTA's run in the global counter, then every
// thread writes its slot.  A 256-thread CTA therefore issues at most NCLS global atomics per 256 paths instead of one per
// warp and class, which matters because all of them hit the same few addresses.  Class k appends to queue0 + k * stride
// and counter0 + k.  Must be called by all threads of the CTA (three barriers; consecutive calls need no fourth: the
// shared words are rewritten only behind the next call's barriers).
template <int NCLS>
__device__ __forceinline__ void block_append(int cls, uint32_t value, uint32_t* __restrict__ queue0, uint32_t stride, uint32_t* __restrict__ counter0)
{
  __shared__ uint32_t sCount[NCLS], sBase[NCLS];
  if (threadIdx.x < NCLS) sCount[threadIdx.x] = 0u;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t peers = 0u;
#pragma unroll
  for (int k = 0; k < NCLS; ++k)
  {
    const uint32_t m = __ballot_sync(0xffffffffu, cls == k);
    if (cls == k) peers = m;
  }
  uint32_t offset = 0;
  const uint32_t leader = peers ? (uint32_t)__ffs((int)peers) - 1u : lane;
  if (peers && lane == leader) offset = atomicAdd(&sCount[cls], (uint32_t)__popc(peers));
  // peers of the same class share their leader's reservation
  offset = __shfl_sync(0xffffffffu, offset, leader) + (uint32_t)__popc(peers & ((1u << lane) - 1u));
  __syncthreads();
  if (threadIdx.x < NCLS && sCount[threadIdx.x]) sBase[threadIdx.x] = atomicAdd(counter0 + threadIdx.x, sCount[threadIdx.x]);
  __syncthreads();
  if (peers) queue0[(size_t)cls * stride + sBase[cls] + offset] = value;
}

// The two appends of the shade kernels behind ONE set of barriers: queue A (paths that continue) and queue B (shadow rays);
// a path may enter both.  Within the CTA's run of each queue the entries are grouped by the direction octant of their ray
// (octA / octB in 0..7): the persistent traversal warps take consecutive queue entries, so a refill mostly brings rays that
// descend the BVH in the same child order.
__device__ __forceinline__ void block_append2_sorted(bool inA, uint32_t octA, uint32_t* __restrict__ queueA, uint32_t* __restrict__ counterA,
                                                     bool inB, uint32_t octB, uint32_t* __restrict__ queueB, uint32_t* __restrict__ counterB, uint32_t value)
{
  __shared__ uint32_t sCount[16], sBase[16];
  if (threadIdx.x < 16) sCount[threadIdx.x] = 0u;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
  uint32_t peersA = 0u, peersB = 0u;
#pragma unroll
  for (uint32_t k = 0; k < 8u; ++k)
  {
    const uint32_t mA = __ballot_sync(0xffffffffu, inA && octA == k), mB = __ballot_sync(0xffffffffu, inB && octB == k);
    if (inA && octA == k) peersA = mA;
    if (inB && octB == k) peersB = mB;
  }
  uint32_t offA = 0, offB = 0;
  const uint32_t leaderA = peersA ? (uint32_t)__ffs((int)peersA) - 1u : lane, leaderB = peersB ? (uint32_t)__ffs((int)peersB) - 1u : lane;
  if (peersA && lane == leaderA) offA = atomicAdd(&sCount[octA], (uint32_t)__popc(peersA));
  if (peersB && lane == leaderB) offB = atomicAdd(&sCount[8u + octB], (uint32_t)__popc(peersB));
  offA = __shfl_sync(0xffffffffu, offA, leaderA) + (uint32_t)__popc(peersA & below);
  offB = __shfl_sync(0xffffffffu, offB, leaderB) + (uint32_t)__popc(peersB & below);
  __syncthreads();
  if (threadIdx.x < 2)     // thread 0: queue A, thread 1: queue B -- one global reservation for the eight octant runs
  {
    const uint32_t first = 8u * threadIdx.x;
    uint32_t total = 0;
#pragma unroll
    for (uint32_t k = 0; k < 8u; ++k) total += sCount[first + k];
    if (total)
    {
      uint32_t base = atomicAdd(threadIdx.x ? counterB : counterA, total);
#pragma unroll
      for (uint32_t k = 0; k < 8u; ++k) { sBase[first + k] = base; base += sCount[first + k]; }
    }
  }
  __syncthreads();
  if (inA) queueA[sBase[octA] + offA] = value;
  if (inB) queueB[sBase[8u + octB] + offB] = value;
}

// Two independent appends (a path may enter both queues) behind ONE set of barriers.
__device__ __forceinline__ void block_append2(bool inA, uint32_t* __restrict__ queueA, uint32_t* __restrict__ counterA,
                                              bool inB, uint32_t* __restrict__ queueB, uint32_t* __restrict__ counterB, uint32_t value)
{
  __shared__ uint32_t sCount[2], sBase[2];
  if (threadIdx.x < 2) sCount[threadIdx.x] = 0u;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31u, below = (1u << lane) - 1u;
  const uint32_t mA = __ballot_sync(0xffffffffu, inA), mB = __ballot_sync(0xffffffffu, inB);
  uint32_t offA = 0, offB = 0;
  if (lane == 0)
  {
    if (mA) offA = atomicAdd(&sCount[0], (uint32_t)__popc(mA));
    if (mB) offB = atomicAdd(&sCount[1], (uint32_t)__popc(mB));
  }
  offA = __shfl_sync(0xffffffffu, offA, 0) + (uint32_t)__popc(mA & below);
  offB = __shfl_sync(0xffffffffu, offB, 0) + (uint32_t)__popc(mB & below);
  __syncthreads();
  if (threadIdx.x == 0 && sCount[0]) sBase[0] = atomicAdd(counterA, sCount[0]);
  if (threadIdx.x == 1 && sCount[1]) sBase[1] = atomicAdd(counterB, sCount[1]);
  __syncthreads();
  if (inA) queueA[sBase[0] + offA] = value;
  if (inB) queueB[sBase[1] + offB] = value;
}

__global__ void __launch_bounds__(kBlock)
k_generate(const __grid_constant__ WfArgs a, uint32_t* __restrict__ queue, uint32_t* __restrict__ count)
{
  const uint32_t pixelsPerIter = a.launchWidth * a.launchHeight;
  const uint32_t n = a.numPaths;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += stride)
  {
    const uint32_t p = base + threadIdx.x;
    bool alive = false;
    if (p < n)
    {
      const uint32_t it = p / pixelsPerIter, idx = p - it * pixelsPerIter;
      uint32_t x, y;
      launch_xy(idx, a.launchWidth, a.launchHeight, x, y);
      uint32_t seed = 0, col = 0; float3 pos, wi;
      alive = start_path(a.sys, a.launchWidth, x, y, a.iterFirst + (int)it, seed, pos, wi, col);
      if (alive)
      {
        a.wf.rayOrg[p] = make_float4(pos.x, pos.y, pos.z, a.sys.sceneEpsilon);
        a.wf.rayDir[p] = make_float4(wi.x, wi.y, wi.z, RT_DEFAULT_MAX);
        a.wf.throughput[p] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
        a.wf.radiance[p] = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(0u));
        a.wf.misc[p] = make_uint4(seed, 0u, (uint32_t)RT_MATERIAL_STACK_EMPTY, col);
      }
      else
      {
        a.wf.misc[p] = make_uint4(0u, 0u, 0u, kNoPixel);
      }
    }
    block_append<1>(alive ? 0 : -1, p, queue, 0u, count);
  }
}

// ---- fused primary path: extend of the first segment without a generate pass ----------------------------------------------
// Ray source of the depth-0 extend: the ray of path i is computed from its launch index at fetch time (start_path: TEA seed,
// jitter, lens shader) instead of being written by k_generate and read back.  It lives in this translation unit because the
// ray must carry the shading arithmetic's bits (-fmad=false); the intersector pins its own rounding with intrinsics and the
// box test only has to be conservative, so the traversal is indifferent to the flag.
struct ExtendPrimary
{
  WfArgs a;
  __device__ __forceinline__ bool load(uint32_t i, float4& o, float4& d, uint32_t& path) const
  {
    path = i;
    const uint32_t pixelsPerIter = a.launchWidth * a.launchHeight;
    const uint32_t it = i / pixelsPerIter, idx = i - it * pixelsPerIter;
    uint32_t x, y;
    launch_xy(idx, a.launchWidth, a.launchHeight, x, y);
    uint32_t seed = 0, col = 0; float3 pos, wi;
    if (!start_path(a.sys, a.launchWidth, x, y, a.iterFirst + (int)it, seed, pos, wi, col))
    {
      a.wf.hitInst[i] = kDeadPath;
      return false;
    }
    o = make_float4(pos.x, pos.y, pos.z, a.sys.sceneEpsilon);
    d = make_float4(wi.x, wi.y, wi.z, RT_DEFAULT_MAX);
    return true;
  }
  __device__ __forceinline__ void store(uint32_t path, const TraceHit& h) const
  {
    __stcs(a.wf.hit + path, make_float4(h.t, h.u, h.v, __uint_as_float(h.prim)));
    __stcs(a.wf.hitInst + path, h.inst);
  }
};

constexpr int kPrimaryBlock = 128;

template <bool COUNT, int TRICAP = 0>
__global__ void __launch_bounds__(kPrimaryBlock, RTC_TRACE_MIN_BLOCKS)
k_extend_primary(const SceneDesc sc, const ExtendPrimary policy, uint32_t n, uint32_t* __restrict__ cursor, unsigned long long* __restrict__ counts)
{
  __shared__ uint2 smem[RTC_SM_STACK * kPrimaryBlock + (RTC_SM_RAY_WORDS * kPrimaryBlock + 1) / 2];
  trace_stream<false, COUNT, kPrimaryBlock, false, TRICAP>(sc, n, cursor, policy, smem, counts);
}

__device__ __forceinline__ float3 xf_vector(const float4 r0, const float4 r1, const float4 r2, float3 v)
{
  return f3(r0.x * v.x + r0.y * v.y + r0.z * v.z, r1.x * v.x + r1.y * v.y + r1.z * v.z, r2.x * v.x + r2.y * v.y + r2.z * v.z);
}
__device__ __forceinline__ float3 xf_normal(const float4 r0, const float4 r1, const float4 r2, float3 v)
{
  return f3(r0.x * v.x + r1.x * v.y + r2.x * v.z, r0.y * v.x + r1.y * v.y + r2.y * v.z, r0.z * v.x + r1.z * v.y + r2.z * v.z);
}
__device__ __forceinline__ float3 ld3(const float* p) { return f3(__ldg(p), __ldg(p + 1), __ldg(p + 2)); }

// Surface classes of the shade stage.  After extend, k_bin sorts the live paths into one queue per class, and a
// specialised instantiation of k_shade runs per class: a warp then executes ONE BSDF (or the miss program) instead of
// serialising all of them, and each instantiation carries only its own code.
enum : int { SHADE_MISS = 0, SHADE_BRDF_DIFFUSE = 1, SHADE_BRDF_SPECULAR = 2, SHADE_BSDF_SPECULAR = 3, SHADE_BRDF_GGX = 4, SHADE_BSDF_GGX = 5,
             SHADE_OTHER = 6, SHADE_NUM_CLASSES = 7 };

// queueIn == nullptr (fused primary path): the queue is the identity over all a.numPaths paths, launch indices outside
// the image carry hitInst == kDeadPath, and the number of live paths is added to *aliveCount (the depth-0 ray count).
__global__ void __launch_bounds__(kBlock)
k_bin(const __grid_constant__ WfArgs a, const SceneDesc sc, const uint32_t* __restrict__ queueIn, const uint32_t* __restrict__ countIn,
      uint32_t* __restrict__ bins, uint32_t binStride, uint32_t* __restrict__ binCounts, uint32_t* __restrict__ aliveCount)
{
  const uint32_t n = queueIn ? *countIn : a.numPaths;
  const uint32_t stride = gridDim.x * blockDim.x;
  const rt_MaterialDefinition* materials = reinterpret_cast<const rt_MaterialDefinition*>(a.sys.materialDefinitions);
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += stride)
  {
    const uint32_t i = base + threadIdx.x;
    int cls = -1; uint32_t p = 0;
    if (i < n)
    {
      p = queueIn ? queueIn[i] : i;
      const uint32_t inst = a.wf.hitInst[p];
      if (inst == 0xffffffffu) cls = SHADE_MISS;
      else if (inst == kDeadPath) cls = -1;
      else
      {
        const int index = materials[sc.geomInst[inst].materialIndex].indexBSDF;
        cls = (0 <= index && index < RT_NUM_BSDF_INDICES) ? 1 + index : SHADE_OTHER;
      }
    }
    block_append<SHADE_NUM_CLASSES>(cls, p, bins, binStride, binCounts);
    if (!queueIn)
    {
      const int alive = __syncthreads_count(cls >= 0);
      if (threadIdx.x == 0 && alive) atomicAdd(aliveCount, (uint32_t)alive);
    }
  }
}

template <int CLASS> SD void bsdf_sample_class(const rt_MaterialDefinition& m, const State& st, Prd& prd)
{
  if (CLASS == SHADE_BRDF_DIFFUSE)        sample_brdf_diffuse(m, st, prd);
  else if (CLASS == SHADE_BRDF_SPECULAR)  sample_brdf_specular(st, prd);
  else if (CLASS == SHADE_BSDF_SPECULAR)  sample_bsdf_specular(m, st, prd);
  else if (CLASS == SHADE_BRDF_GGX)       sample_brdf_ggx(m, st, prd);
  else if (CLASS == SHADE_BSDF_GGX)       sample_bsdf_ggx(m, st, prd);
  else                                    bsdf_sample(m, st, prd);
}
template <int CLASS> SD float4 bsdf_eval_class(const rt_MaterialDefinition& m, const State& st, const Prd& prd, float3 wiL)
{
  if (CLASS == SHADE_BRDF_DIFFUSE)  return eval_brdf_diffuse(st, wiL);
  if (CLASS == SHADE_BRDF_GGX)      return eval_brdf_ggx(m, st, prd, wiL);
  if (CLASS == SHADE_OTHER)         return bsdf_eval(m, st, prd, wiL);
  return make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

// TEX = false: the kernels of scenes without material textures (every configuration of BASELINE.json).
// TEX = true : interpolates the texture coordinates and modulates the albedo (closesthit.cu:233-240); with deferRR the
//              Russian roulette of a path that casts a shadow ray is left to k_cutout_shadow, because the shadow ray's
//              any-hit programs draw from the path's seed BEFORE the integrator does (closesthit.cu:281 precedes
//              raygeneration.cu:111).
// PRIMARY = true (fused primary path, first segment only): there is no generate pass; the path's seed, ray and pixel are
//              recomputed from the launch index instead of being read back, throughput is 1 and radiance 0.
template <int CLASS, bool TEX, bool PRIMARY>
__global__ void __launch_bounds__(kBlock)
k_shade(const __grid_constant__ WfArgs a, const SceneDesc sc,
        const uint32_t* __restrict__ queueIn, const uint32_t* __restrict__ countIn,
        uint32_t* __restrict__ queueOut, uint32_t* __restrict__ countOut,
        uint32_t* __restrict__ shadowQueue, uint32_t* __restrict__ shadowCount, const int deferRR)
{
  const rt_SystemData& sys = a.sys;
  const uint32_t n = *countIn;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += stride)
  {
    const uint32_t i = base + threadIdx.x;
    if (CLASS == SHADE_MISS)
    {
      // A path that left the scene ends here (the miss programs set FLAG_TERMINATE): it touches its throughput, its radiance and
      // its volume-stack index, the ray direction only for the spherical environment -- not the ray origin, the hit record or
      // the seed -- and joins no queue, so this instantiation has no barrier.  Same operations as the general path below.
      if (i < n)
      {
        const uint32_t pm = queueIn[i];
        float4 tpm, Lfm; float3 wim = f3(0.0f, 0.0f, 1.0f); int stackIdxM;
        if (PRIMARY)
        {
          tpm = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
          Lfm = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(0u));
          stackIdxM = RT_MATERIAL_STACK_EMPTY;
          if (a.miss == RT_MISS_SPHERE)
          {
            const uint32_t pixelsPerIter = a.launchWidth * a.launchHeight;
            const uint32_t it = pm / pixelsPerIter, idx = pm - it * pixelsPerIter;
            uint32_t x, y;
            launch_xy(idx, a.launchWidth, a.launchHeight, x, y);
            uint32_t seed = 0, col = 0; float3 pos;
            start_path(sys, a.launchWidth, x, y, a.iterFirst + (int)it, seed, pos, wim, col);
          }
        }
        else
        {
          tpm = a.wf.throughput[pm];
          Lfm = a.wf.radiance[pm];
          stackIdxM = (int)a.wf.misc[pm].z;
          if (a.miss == RT_MISS_SPHERE) { const float4 rd = a.wf.rayDir[pm]; wim = f3(rd.x, rd.y, rd.z); }
        }
        Prd prd;
        prd.wi = wim;
        prd.pdf = tpm.w;
        prd.flags = __float_as_uint(Lfm.w) & RT_FLAG_CLEAR_MASK;
        prd.sigma_t = f3(0.0f);
        prd.distance = RT_DEFAULT_MAX;
        if (RT_MATERIAL_STACK_FIRST <= stackIdxM)
        {
          const float4 top = a.wf.absStack[(size_t)pm * 4 + stackIdxM];
          prd.flags |= RT_FLAG_VOLUME;
          prd.sigma_t = f3(top.x, top.y, top.z);
        }
        miss_program(sys, a.miss, prd);
        float3 throughput = f3(tpm.x, tpm.y, tpm.z);
        if (prd.flags & RT_FLAG_VOLUME)
          throughput = throughput * f3(rt_expf(-prd.distance * prd.sigma_t.x), rt_expf(-prd.distance * prd.sigma_t.y), rt_expf(-prd.distance * prd.sigma_t.z));
        const float3 radiance = f3(Lfm.x, Lfm.y, Lfm.z) + throughput * prd.radiance;
        a.wf.radiance[pm] = make_float4(radiance.x, radiance.y, radiance.z, __uint_as_float(prd.flags));
      }
      continue;
    }
    bool continues = false, shadow = false, pendingRR = false;
    uint32_t p = 0, octContinue = 0, octShadow = 0;
    if (i < n)
    {
      p = queueIn[i];
      float4 ro, rd, tp, Lf; uint4 misc;
      if (PRIMARY)
      {
        const uint32_t pixelsPerIter = a.launchWidth * a.launchHeight;
        const uint32_t it = p / pixelsPerIter, idx = p - it * pixelsPerIter;
        uint32_t x, y;
        launch_xy(idx, a.launchWidth, a.launchHeight, x, y);
        uint32_t seed = 0, col = 0; float3 pos, wi;
        start_path(sys, a.launchWidth, x, y, a.iterFirst + (int)it, seed, pos, wi, col);     // alive: k_bin dropped the others
        ro = make_float4(pos.x, pos.y, pos.z, sys.sceneEpsilon);
        rd = make_float4(wi.x, wi.y, wi.z, RT_DEFAULT_MAX);
        tp = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
        Lf = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(0u));
        misc = make_uint4(seed, 0u, (uint32_t)RT_MATERIAL_STACK_EMPTY, col);
      }
      else
      {
        ro = a.wf.rayOrg[p]; rd = a.wf.rayDir[p];
        tp = a.wf.throughput[p];
        Lf = a.wf.radiance[p];
        misc = a.wf.misc[p];
      }
      const float4 hit = a.wf.hit[p];
      const uint32_t hitInst = a.wf.hitInst[p];

      Prd prd;
      prd.pos = f3(ro.x, ro.y, ro.z);
      prd.wi = f3(rd.x, rd.y, rd.z);
      prd.seed = misc.x;
      int depth = TEX ? (int)(misc.y & kDepthMask) : (int)misc.y;
      int stackIdx = (int)misc.z;
      float3 throughput = f3(tp.x, tp.y, tp.z);
      float3 radiance = f3(Lf.x, Lf.y, Lf.z);
      prd.pdf = tp.w;
      prd.flags = __float_as_uint(Lf.w);
      prd.f_over_pdf = f3(0.0f);
      prd.absorption_ior = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
      prd.sigma_t = f3(0.0f);

      // ---- per-segment reset (raygeneration.cu:63-78)
      prd.wo = -prd.wi;
      prd.ior = make_float2(1.0f, 1.0f);
      prd.distance = RT_DEFAULT_MAX;
      prd.flags &= RT_FLAG_CLEAR_MASK;
      if (RT_MATERIAL_STACK_FIRST <= stackIdx)
      {
        const float4 top = a.wf.absStack[(size_t)p * 4 + stackIdx];
        prd.flags |= RT_FLAG_VOLUME;
        prd.sigma_t = f3(top.x, top.y, top.z);
        prd.ior.x = top.w;
        if (RT_MATERIAL_STACK_FIRST <= stackIdx - 1) prd.ior.y = a.wf.absStack[(size_t)p * 4 + stackIdx - 1].w;
      }

      if (CLASS == SHADE_MISS)
      {
        miss_program(sys, a.miss, prd);
      }
      else
      {
        // ---- __closesthit__radiance (closesthit.cu:126-305)
        const rt_GeometryInstanceData gi = sc.geomInst[hitInst];
        const uint32_t prim = __float_as_uint(hit.w);
        const uint32_t* ix = reinterpret_cast<const uint32_t*>(gi.indices) + 3u * (size_t)prim;
        const uint32_t i0 = __ldg(ix), i1 = __ldg(ix + 1), i2 = __ldg(ix + 2);
        // TriangleAttributes = 48 bytes = three 16-byte loads per vertex: vertex.xyz|tangent.x, tangent.yz|normal.xy, normal.z|texcoord.xyz
        const float4* V0 = reinterpret_cast<const float4*>(gi.attributes) + 3u * (size_t)i0;
        const float4* V1 = reinterpret_cast<const float4*>(gi.attributes) + 3u * (size_t)i1;
        const float4* V2 = reinterpret_cast<const float4*>(gi.attributes) + 3u * (size_t)i2;
        const float4 a00 = __ldg(V0), a01 = __ldg(V0 + 1), a02 = __ldg(V0 + 2);
        const float4 a10 = __ldg(V1), a11 = __ldg(V1 + 1), a12 = __ldg(V1 + 2);
        const float4 a20 = __ldg(V2), a21 = __ldg(V2 + 1), a22 = __ldg(V2 + 2);
        const float bx = hit.y, by = hit.z;
        const float alpha = 1.0f - bx - by;
        const float3 p0 = f3(a00.x, a00.y, a00.z), p1 = f3(a10.x, a10.y, a10.z), p2 = f3(a20.x, a20.y, a20.z);
        const float3 ng = cross(p1 - p0, p2 - p0);
        const float3 tg = f3(a00.w, a01.x, a01.y) * alpha + f3(a10.w, a11.x, a11.y) * bx + f3(a20.w, a21.x, a21.y) * by;
        const float3 ns = f3(a01.z, a01.w, a02.x) * alpha + f3(a11.z, a11.w, a12.x) * bx + f3(a21.z, a21.w, a22.x) * by;

        const float4* o2w = sc.objectToWorld + (size_t)hitInst * 3u;
        const float4* w2o = sc.instances + (size_t)hitInst * 4u;
        const float4 w0 = __ldg(o2w), w1 = __ldg(o2w + 1), w2 = __ldg(o2w + 2);
        const float4 v0 = __ldg(w2o), v1 = __ldg(w2o + 1), v2 = __ldg(w2o + 2);

        State state;
        state.normalGeo = normalize(xf_normal(v0, v1, v2, ng));
        state.tangent   = normalize(xf_vector(w0, w1, w2, tg));
        state.normal    = normalize(xf_normal(v0, v1, v2, ns));

        prd.distance = hit.x;
        prd.pos = prd.pos + prd.wi * prd.distance;
        prd.flags |= (0.0f <= dot(prd.wo, state.normalGeo)) ? RT_FLAG_FRONTFACE : 0u;
        if ((prd.flags & RT_FLAG_FRONTFACE) == 0u)
        {
          state.normalGeo = -state.normalGeo;
          state.tangent = -state.tangent;
          state.normal = -state.normal;
        }
        prd.radiance = f3(0.0f);

        bool emissive = false;
        if (0 <= gi.lightIndex && (prd.flags & RT_FLAG_FRONTFACE))
        {
          const float cosTheta = dot(prd.wo, state.normalGeo);
          if (RT_DENOMINATOR_EPSILON < cosTheta)
          {
            const rt_LightDefinition& light = reinterpret_cast<const rt_LightDefinition*>(sys.lightDefinitions)[gi.lightIndex];
            float3 emission = f3(light.emission);
            const float lightPdf = (prd.distance * prd.distance) / (light.area * cosTheta);
            if ((prd.flags & RT_FLAG_DIFFUSE) && RT_DENOMINATOR_EPSILON < lightPdf)
              emission = emission * power_heuristic(prd.pdf, lightPdf);
            prd.radiance = emission;
            prd.flags |= RT_FLAG_TERMINATE;
            emissive = true;
          }
        }
        if (!emissive)
        {
          prd.f_over_pdf = f3(0.0f);
          prd.pdf = 0.0f;
          const rt_MaterialDefinition material = reinterpret_cast<const rt_MaterialDefinition*>(sys.materialDefinitions)[gi.materialIndex];
          state.albedo = f3(material.albedo);
          if (TEX && material.textureAlbedo != 0)
          {
            const float3 texcoord = f3(a02.y, a02.z, a02.w) * alpha + f3(a12.y, a12.z, a12.w) * bx + f3(a22.y, a22.z, a22.w) * by;
            state.albedo = state.albedo * tex2d_wrap(material.textureAlbedo, texcoord.x, texcoord.y);
          }
          prd.flags = (prd.flags & ~RT_FLAG_DIFFUSE) | RT_FLAG_HIT | material.flags;
          bsdf_sample_class<CLASS>(material, state, prd);

          const int numLights = sys.numLights;
          // only the diffuse and glossy-reflection lobes ever set FLAG_DIFFUSE: the specular classes carry no NEE code
          if ((CLASS == SHADE_BRDF_DIFFUSE || CLASS == SHADE_BRDF_GGX || CLASS == SHADE_OTHER) && (prd.flags & RT_FLAG_DIFFUSE) && 0 < numLights)
          {
            const float2 sample = rng2(prd.seed);
            LightSample ls; ls.pdf = 0.0f; ls.distance = 0.0f; ls.direction = f3(0.0f); ls.emission = f3(0.0f);
            if (1 < numLights)
            {
              int idx = (int)floorf(rng(prd.seed) * (float)numLights);
              idx = idx < 0 ? 0 : (idx > numLights - 1 ? numLights - 1 : idx);
              ls.index = idx;
            }
            else ls.index = 0;
            const int type = reinterpret_cast<const rt_LightDefinition*>(sys.lightDefinitions)[ls.index].type;
            if (type == RT_LIGHT_PARALLELOGRAM) light_parallelogram(sys, prd.pos, sample, ls);
            else if (a.miss == RT_MISS_SPHERE)  light_env_sphere(sys, sample, ls);
            else                                light_env_constant(numLights, sample, ls);
            if (0.0f < ls.pdf)
            {
              const float4 bp = bsdf_eval_class<CLASS>(material, state, prd, ls.direction);
              const float3 f = f3(bp.x, bp.y, bp.z);
              if (0.0f < bp.w && !is_null(f))
              {
                // the shadow ray is traced by `connect`; its contribution is what closesthit.cu:289-299 would add
                // if the ray is unoccluded, already multiplied by the throughput the integrator applies at :100
                if (prd.flags & RT_FLAG_VOLUME)
                  ls.emission = ls.emission * f3(rt_expf(-ls.distance * prd.sigma_t.x), rt_expf(-ls.distance * prd.sigma_t.y), rt_expf(-ls.distance * prd.sigma_t.z));
                const float weightMis = power_heuristic(ls.pdf, bp.w);
                const float3 c = f * ls.emission * (weightMis * dot(ls.direction, state.normal) / ls.pdf);
                float3 tseg = throughput;
                if (prd.flags & RT_FLAG_VOLUME)
                  tseg = tseg * f3(rt_expf(-prd.distance * prd.sigma_t.x), rt_expf(-prd.distance * prd.sigma_t.y), rt_expf(-prd.distance * prd.sigma_t.z));
                const float3 tc = tseg * c;
                a.wf.shadowOrg[p] = make_float4(prd.pos.x, prd.pos.y, prd.pos.z, sys.sceneEpsilon);
                a.wf.shadowDir[p] = make_float4(ls.direction.x, ls.direction.y, ls.direction.z, ls.distance - sys.sceneEpsilon);
                a.wf.shadowContrib[p] = make_float4(tc.x, tc.y, tc.z, 0.0f);
                octShadow = ((ls.direction.x < 0.0f) ? 4u : 0u) | ((ls.direction.y < 0.0f) ? 2u : 0u) | ((ls.direction.z < 0.0f) ? 1u : 0u);
                shadow = true;
              }
            }
          }
        }
      }

      // ---- integrator epilogue (raygeneration.cu:92-145)
      if (prd.flags & RT_FLAG_VOLUME)
        throughput = throughput * f3(rt_expf(-prd.distance * prd.sigma_t.x), rt_expf(-prd.distance * prd.sigma_t.y), rt_expf(-prd.distance * prd.sigma_t.z));
      radiance = radiance + throughput * prd.radiance;

      bool ended = (prd.flags & RT_FLAG_TERMINATE) || prd.pdf <= 0.0f || is_null(prd.f_over_pdf);
      if (!ended)
      {
        throughput = throughput * prd.f_over_pdf;
        if (sys.pathLengths.x <= depth)
        {
          if (TEX && deferRR && shadow) pendingRR = true;
          else
          {
            const float probability = fmax3(throughput);
            if (probability < rng(prd.seed)) ended = true;
            else throughput = divs(throughput, probability);
          }
        }
      }
      if (!ended)
      {
        if ((prd.flags & (RT_FLAG_THINWALLED | RT_FLAG_TRANSMISSION)) == RT_FLAG_TRANSMISSION)
        {
          if (prd.flags & RT_FLAG_FRONTFACE)
          {
            stackIdx = (stackIdx + 1 < RT_MATERIAL_STACK_LAST) ? stackIdx + 1 : RT_MATERIAL_STACK_LAST;
            a.wf.absStack[(size_t)p * 4 + stackIdx] = prd.absorption_ior;
          }
          else
          {
            stackIdx = (stackIdx - 1 > RT_MATERIAL_STACK_EMPTY) ? stackIdx - 1 : RT_MATERIAL_STACK_EMPTY;
          }
        }
        ++depth;
        continues = depth < sys.pathLengths.y;
      }
      if (!continues) pendingRR = false;      // the path ends here whatever the roulette says: its draw cannot matter

      a.wf.radiance[p] = make_float4(radiance.x, radiance.y, radiance.z, __uint_as_float(prd.flags));
      if (continues)
      {
        a.wf.rayOrg[p] = make_float4(prd.pos.x, prd.pos.y, prd.pos.z, sys.sceneEpsilon);
        a.wf.rayDir[p] = make_float4(prd.wi.x, prd.wi.y, prd.wi.z, RT_DEFAULT_MAX);
        octContinue = ((prd.wi.x < 0.0f) ? 4u : 0u) | ((prd.wi.y < 0.0f) ? 2u : 0u) | ((prd.wi.z < 0.0f) ? 1u : 0u);
        a.wf.throughput[p] = make_float4(throughput.x, throughput.y, throughput.z, prd.pdf);
        misc.x = prd.seed; misc.y = (uint32_t)depth | (pendingRR ? kPendingRR : 0u); misc.z = (uint32_t)stackIdx;
        a.wf.misc[p] = misc;
      }
      else if (TEX && deferRR && shadow)
      {
        // the shadow ray's any-hit programs draw from this seed (k_cutout_shadow)
        misc.x = prd.seed; misc.y = (uint32_t)depth;
        a.wf.misc[p] = misc;
      }
    }
    // a path whose roulette is pending is appended to the next queue by k_cutout_shadow once its shadow ray is resolved
    block_append2_sorted(continues && !pendingRR, octContinue, queueOut, countOut, shadow, octShadow, shadowQueue, shadowCount, p);
  }
}

// ---- ordered any-hit processing of cutout materials (anyhit.cu:46-80, :94-132) --------------------------------------------
// Candidates of a ray are presented closest first (canonical order (t, instance, primitive)); the kernels below play the
// any-hit program on the candidate in hit[p] / hitInst[p] and queue the path for a re-trace past it when it is ignored.

// opacity of the candidate of path p; false when the instance's hit records have no cutout program or no texture is bound
SD bool cutout_candidate(const WfArgs& a, const SceneDesc& sc, uint32_t inst, const float4 hit, bool& cutoutRecords, float& opacity)
{
  cutoutRecords = (__ldg(sc.instFlags + inst) & RTC_INSTANCE_CUTOUT) != 0u;
  if (!cutoutRecords) return false;
  const rt_GeometryInstanceData gi = sc.geomInst[inst];
  const uint64_t texture = reinterpret_cast<const rt_MaterialDefinition*>(a.sys.materialDefinitions)[gi.materialIndex].textureCutout;
  if (texture == 0) return false;
  const uint32_t prim = __float_as_uint(hit.w);
  const uint32_t* ix = reinterpret_cast<const uint32_t*>(gi.indices) + 3u * (size_t)prim;
  const uint32_t i0 = __ldg(ix), i1 = __ldg(ix + 1), i2 = __ldg(ix + 2);
  const float* A0 = reinterpret_cast<const float*>(gi.attributes) + 12u * (size_t)i0;
  const float* A1 = reinterpret_cast<const float*>(gi.attributes) + 12u * (size_t)i1;
  const float* A2 = reinterpret_cast<const float*>(gi.attributes) + 12u * (size_t)i2;
  const float bx = hit.y, by = hit.z;
  const float alpha = 1.0f - bx - by;
  const float3 texcoord = ld3(A0 + 9) * alpha + ld3(A1 + 9) * bx + ld3(A2 + 9) * by;
  opacity = intensity3(tex2d_wrap(texture, texcoord.x, texcoord.y));
  return true;
}

// __anyhit__radiance_cutout on the closest candidate of every path in queueIn; ignored -> queueOut (re-trace past it)
__global__ void __launch_bounds__(kBlock)
k_cutout_radiance(const __grid_constant__ WfArgs a, const SceneDesc sc, const uint32_t* __restrict__ queueIn, const uint32_t* __restrict__ countIn,
                  uint32_t* __restrict__ queueOut, uint32_t* __restrict__ countOut)
{
  const uint32_t n = *countIn;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += stride)
  {
    const uint32_t i = base + threadIdx.x;
    bool again = false; uint32_t p = 0;
    if (i < n)
    {
      p = queueIn[i];
      const uint32_t inst = a.wf.hitInst[p];
      bool records; float opacity;
      if (inst != 0xffffffffu && cutout_candidate(a, sc, inst, a.wf.hit[p], records, opacity) && opacity < 1.0f)
      {
        uint32_t seed = a.wf.misc[p].x;
        again = opacity <= rng(seed);          // optixIgnoreIntersection
        a.wf.misc[p].x = seed;
      }
    }
    block_append<1>(again ? 0 : -1, p, queueOut, 0u, countOut);
  }
}

// __anyhit__shadow / __anyhit__shadow_cutout on the closest candidate of every shadow ray in queueIn.  No candidate left: the
// light is visible, the contribution is added (closesthit.cu:289-299).  Ignored: queueOut (re-trace past it).  Once the ray
// is resolved, a postponed Russian roulette is played and the survivor appended to the next extend queue.
// where the survivors of a postponed Russian roulette go (the next depth's extend queue); device-resident so that the
// kernels of the any-hit rounds have the same arguments at every depth (they are replayed from a CUDA graph)
struct CutoutNext { uint32_t* queue; uint32_t* count; };

__global__ void k_set_cutout_next(CutoutNext* next, uint32_t* queue, uint32_t* count) { next->queue = queue; next->count = count; }

// loop condition of the any-hit rounds: another round is needed while the last one ignored a candidate
__global__ void k_cutout_condition(cudaGraphConditionalHandle handle, const uint32_t* __restrict__ ignored)
{
  cudaGraphSetConditional(handle, *ignored != 0u ? 1u : 0u);
}

__global__ void __launch_bounds__(kBlock)
k_cutout_shadow(const __grid_constant__ WfArgs a, const SceneDesc sc, const uint32_t* __restrict__ queueIn, const uint32_t* __restrict__ countIn,
                uint32_t* __restrict__ queueOut, uint32_t* __restrict__ countOut, const CutoutNext* __restrict__ next)
{
  uint32_t* __restrict__ queueNext = next->queue;
  uint32_t* __restrict__ countNext = next->count;
  const uint32_t n = *countIn;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += stride)
  {
    const uint32_t i = base + threadIdx.x;
    bool again = false, survives = false; uint32_t p = 0;
    if (i < n)
    {
      p = queueIn[i];
      const uint32_t inst = a.wf.hitInst[p];
      uint4 misc = a.wf.misc[p];
      const uint32_t seedIn = misc.x, flagsIn = misc.y;
      if (inst == 0xffffffffu)
      {
        const float4 c = a.wf.shadowContrib[p];
        float4 L = a.wf.radiance[p];
        L.x = L.x + c.x; L.y = L.y + c.y; L.z = L.z + c.z;
        a.wf.radiance[p] = L;
      }
      else
      {
        bool records; float opacity = 1.0f;
        cutout_candidate(a, sc, inst, a.wf.hit[p], records, opacity);
        if (records && opacity < 1.0f) again = opacity <= rng(misc.x);
        // else: FLAG_SHADOW, optixTerminateRay
      }
      if (!again && (misc.y & kPendingRR))
      {
        misc.y &= ~kPendingRR;
        float4 tp = a.wf.throughput[p];
        const float3 throughput = f3(tp.x, tp.y, tp.z);
        const float probability = fmax3(throughput);
        if (!(probability < rng(misc.x)))
        {
          const float3 t = divs(throughput, probability);
          a.wf.throughput[p] = make_float4(t.x, t.y, t.z, tp.w);
          survives = true;
        }
      }
      if (misc.x != seedIn || misc.y != flagsIn) a.wf.misc[p] = misc;
    }
    block_append2(again, queueOut, countOut, survives, queueNext, countNext, p);
  }
}

// One thread per launch index; applies the batch's iterations in order (running average is order dependent).
__global__ void __launch_bounds__(kBlock)
k_accumulate(const __grid_constant__ WfArgs a)
{
  const uint32_t pixelsPerIter = a.launchWidth * a.launchHeight;
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= pixelsPerIter) return;
  uint32_t x, y;
  launch_xy(idx, a.launchWidth, a.launchHeight, x, y);
  uint32_t col = x;      // raygeneration.cu:178-186: the pixel column of this launch index, nothing to do outside the image
  if (a.sys.distribution && 1 < a.sys.deviceCount)
  {
    col = distribute(a.sys, x, y);
    if ((uint32_t)a.sys.resolution.x <= col) return;
  }
  float4* buffer; size_t index;
  if (a.raygen == RTC_RAYGEN_LOCAL_COPY) { buffer = reinterpret_cast<float4*>(a.sys.texelBuffer); index = (size_t)y * a.launchWidth + x; }
  else { buffer = reinterpret_cast<float4*>(a.sys.outputBuffer); index = (size_t)y * (size_t)a.sys.resolution.x + col; }
  float4 dst = buffer[index];
  bool wrote = false;
  for (int b = 0; b < a.iterCount; ++b)
  {
    const float4 L = a.wf.radiance[(size_t)b * pixelsPerIter + idx];
    float3 r = f3(L.x, L.y, L.z);
    if (isnan(r.x) || isnan(r.y) || isnan(r.z)) continue;
    const int it = a.accumFirst + b;
    if (0 < it)
    {
      const float t = 1.0f / (float)(it + 1);
      r = f3(dst.x + t * (r.x - dst.x), dst.y + t * (r.y - dst.y), dst.z + t * (r.z - dst.z));
    }
    dst = make_float4(r.x, r.y, r.z, 1.0f);
    wrote = true;
  }
  if (wrote) buffer[index] = dst;
}

__global__ void __launch_bounds__(kBlock)
k_generate_primary(const __grid_constant__ rt_SystemData sys, uint32_t w, uint32_t h, int iteration, float4* __restrict__ rays)
{
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= w * h) return;
  const uint32_t y = idx / w, x = idx - y * w;
  uint32_t seed, col; float3 pos, wi;
  if (start_path(sys, w, x, y, iteration, seed, pos, wi, col))
  {
    rays[2 * (size_t)idx] = make_float4(pos.x, pos.y, pos.z, sys.sceneEpsilon);
    rays[2 * (size_t)idx + 1] = make_float4(wi.x, wi.y, wi.z, RT_DEFAULT_MAX);
  }
  else
  {
    rays[2 * (size_t)idx] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    rays[2 * (size_t)idx + 1] = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
  }
}

// compositor.cu:38-65
__global__ void __launch_bounds__(kBlock)
k_composite(const __grid_constant__ rt_CompositorData a)
{
  const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t y = blockIdx.y;
  if (x >= (uint32_t)a.launchWidth || y >= (uint32_t)a.resolution.y) return;
  const uint32_t xBlock = x >> a.tileShift.x, yBlock = y >> a.tileShift.y;
  const uint32_t xTile = xBlock * (uint32_t)a.deviceCount + (((uint32_t)a.deviceIndex + yBlock) % (uint32_t)a.deviceCount);
  const uint32_t xPixel = xTile * (uint32_t)a.tileSize.x + (x & (uint32_t)(a.tileSize.x - 1));
  if (xPixel < (uint32_t)a.resolution.x)
  {
    const float4* src = reinterpret_cast<const float4*>(a.tileBuffer);
    float4* dst = reinterpret_cast<float4*>(a.outputBuffer);
    dst[(size_t)y * (size_t)a.resolution.x + xPixel] = src[(size_t)y * (size_t)a.launchWidth + x];
  }
}

// Application.cpp:2262-2295
__global__ void __launch_bounds__(kBlock)
k_tonemap(const __grid_constant__ rt_TonemapperParams p, const float4* __restrict__ rgba, uint8_t* __restrict__ rgb, uint64_t n)
{
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float invGamma = 1.0f / p.gamma;
  const float3 colorBalance = f3(p.colorBalance[0], p.colorBalance[1], p.colorBalance[2]);
  const float invWhitePoint = p.brightness / p.whitePoint;
  const float crushBlacks = p.crushBlacks + p.crushBlacks + 1.0f;
  const float3 lumw = f3(0.3f, 0.59f, 0.11f);
  const float4 px = rgba[i];
  const float3 hdr = f3(px.x, px.y, px.z);
  float3 ldr = (colorBalance * invWhitePoint) * hdr;
  const float3 num = ldr * p.burnHighlights + f3(1.0f), den = ldr + f3(1.0f);
  ldr = ldr * f3(num.x / den.x, num.y / den.y, num.z / den.z);
  float lum = dot(ldr, lumw);
  ldr = f3(lum) + (ldr - f3(lum)) * p.saturation;
  ldr = f3(fmaxf(0.0f, ldr.x), fmaxf(0.0f, ldr.y), fmaxf(0.0f, ldr.z));
  lum = dot(ldr, lumw);
  if (lum < 1.0f)
  {
    const float3 crushed = f3(rt_powf(ldr.x, crushBlacks), rt_powf(ldr.y, crushBlacks), rt_powf(ldr.z, crushBlacks));
    ldr = crushed + (ldr - crushed) * sqrtf(lum);
    ldr = f3(fmaxf(0.0f, ldr.x), fmaxf(0.0f, ldr.y), fmaxf(0.0f, ldr.z));
  }
  float c[3] = { rt_powf(ldr.x, invGamma), rt_powf(ldr.y, invGamma), rt_powf(ldr.z, invGamma) };
#pragma unroll
  for (int k = 0; k < 3; ++k)
  {
    float v = c[k];
    if (v < 0.0f) v = 0.0f;
    if (v > 1.0f) v = 1.0f;
    rgb[3 * i + k] = (uint8_t)(v * 255.0f);
  }
}

} // namespace

// *outOfMemory (optional) tells the caller that the failure was the allocation itself, so it can retry with a smaller batch.
int ensure_wavefront(rtc_context* ctx, uint64_t capacity, bool* outOfMemory)
{
  WavefrontBuffers& wf = ctx->wf;
  if (outOfMemory) *outOfMemory = false;
  if (wf.capacity >= capacity) return 0;
  if (wf.base)
  {
    // The any-hit graph holds pointers into both allocations.  The reset below also forgets the any-hit scratch queues, so they
    // are freed here rather than leaked; they grow with the batch anyway.
    RTC_CUDA(cudaStreamSynchronize(ctx->stream));
    release_cutout_graph(ctx);
    RTC_CUDA(cudaFree(wf.base));
    if (wf.cutBase) RTC_CUDA(cudaFree(wf.cutBase));
    wf = WavefrontBuffers();
  }
  // one allocation, carved into 256-byte aligned SoA arrays
  auto align = [](uint64_t v) { return (v + 255u) & ~(uint64_t)255u; };
  const uint64_t n = capacity;
  uint64_t off = 0;
  const uint64_t oRayOrg = off; off += align(16 * n);
  const uint64_t oRayDir = off; off += align(16 * n);
  const uint64_t oHit = off; off += align(16 * n);
  const uint64_t oHitInst = off; off += align(4 * n);
  const uint64_t oThroughput = off; off += align(16 * n);
  const uint64_t oRadiance = off; off += align(16 * n);
  const uint64_t oMisc = off; off += align(16 * n);
  const uint64_t oAbs = off; off += align(64 * n);
  const uint64_t oSOrg = off; off += align(16 * n);
  const uint64_t oSDir = off; off += align(16 * n);
  const uint64_t oSCon = off; off += align(16 * n);
  const uint64_t oQA = off; off += align(4 * n);
  const uint64_t oQB = off; off += align(4 * n);
  const uint64_t oQS = off; off += align(4 * n);
  const uint64_t oBins = off; off += align(4 * n) * SHADE_NUM_CLASSES;
  const uint64_t oCnt = off; off += align(4 * kNumCounters);
  void* base = nullptr;
  {
    const cudaError_t e = cudaMalloc(&base, off);
    if (e == cudaErrorMemoryAllocation && outOfMemory) { *outOfMemory = true; cudaGetLastError(); }      // clear the sticky error: the caller retries
    if (e != cudaSuccess) return rtc_set_error(__FILE__, __LINE__, "cudaMalloc(wavefront state)", (int)e, cudaGetErrorString(e));
  }
  char* b = static_cast<char*>(base);
  wf.base = base; wf.capacity = capacity;
  wf.rayOrg = (float4*)(b + oRayOrg); wf.rayDir = (float4*)(b + oRayDir); wf.hit = (float4*)(b + oHit); wf.hitInst = (uint32_t*)(b + oHitInst);
  wf.throughput = (float4*)(b + oThroughput); wf.radiance = (float4*)(b + oRadiance); wf.misc = (uint4*)(b + oMisc); wf.absStack = (float4*)(b + oAbs);
  wf.shadowOrg = (float4*)(b + oSOrg); wf.shadowDir = (float4*)(b + oSDir); wf.shadowContrib = (float4*)(b + oSCon);
  wf.queueA = (uint32_t*)(b + oQA); wf.queueB = (uint32_t*)(b + oQB); wf.shadowQueue = (uint32_t*)(b + oQS); wf.counters = (uint32_t*)(b + oCnt);
  wf.bins = (uint32_t*)(b + oBins); wf.binStride = (uint32_t)(align(4 * n) / 4);
  return 0;
}

namespace {

// sums the per-depth queue counts of one batch into the 64-bit statistics
__global__ void k_stats(const uint32_t* __restrict__ counters, int maxDepth, uint32_t numPaths, uint64_t* __restrict__ stats)
{
  if (threadIdx.x == 0 && blockIdx.x == 0)
  {
    uint64_t rad = 0, sh = 0;
    for (int d = 0; d < maxDepth; ++d) { rad += counters[d]; sh += counters[64 + d]; }
    stats[0] += rad; stats[1] += sh; stats[2] += counters[0];
  }
}

} // namespace

namespace {

template <int CLASS>
void launch_shade_class(rtc_context* ctx, cudaStream_t stream, int grid, const WfArgs& a, const SceneDesc& sc, uint32_t* bins, uint32_t binStride, uint32_t* binCounts,
                        uint32_t* qOut, uint32_t* countOut, uint32_t* shadowQueue, uint32_t* shadowCount, bool tex, bool deferRR, bool primary)
{
  if (tex)          k_shade<CLASS, true, false><<<grid, kBlock, 0, stream>>>(a, sc, bins + (size_t)CLASS * binStride, binCounts + CLASS, qOut, countOut, shadowQueue, shadowCount, deferRR ? 1 : 0);
  else if (primary) k_shade<CLASS, false, true><<<grid, kBlock, 0, stream>>>(a, sc, bins + (size_t)CLASS * binStride, binCounts + CLASS, qOut, countOut, shadowQueue, shadowCount, 0);
  else              k_shade<CLASS, false, false><<<grid, kBlock, 0, stream>>>(a, sc, bins + (size_t)CLASS * binStride, binCounts + CLASS, qOut, countOut, shadowQueue, shadowCount, 0);
}

// The seven class kernels of one depth only share the output queues (atomic appends): the diffuse class, the largest, stays on
// the context stream, the other six fork onto side streams after k_bin and join before the next stage, so the small ones fill
// the tails of the large ones instead of each running alone.
int launch_shade_classes(rtc_context* ctx, int grid, const WfArgs& a, const SceneDesc& sc, uint32_t* bins, uint32_t binStride, uint32_t* binCounts,
                         uint32_t* qOut, uint32_t* countOut, uint32_t* shadowQueue, uint32_t* shadowCount, bool tex, bool deferRR, bool primary)
{
  if (!ctx->shadeFork)
  {
    RTC_CUDA(cudaEventCreateWithFlags(&ctx->shadeFork, cudaEventDisableTiming));
    for (int k = 0; k < 6; ++k)
    {
      RTC_CUDA(cudaStreamCreateWithFlags(&ctx->shadeStreams[k], cudaStreamNonBlocking));
      RTC_CUDA(cudaEventCreateWithFlags(&ctx->shadeJoin[k], cudaEventDisableTiming));
    }
  }
  RTC_CUDA(cudaEventRecord(ctx->shadeFork, ctx->stream));
  cudaStream_t s[7];
  int side = 0;
  for (int k = 0; k < 7; ++k)
  {
    if (k == SHADE_BRDF_DIFFUSE) { s[k] = ctx->stream; continue; }
    s[k] = ctx->shadeStreams[side++];
    RTC_CUDA(cudaStreamWaitEvent(s[k], ctx->shadeFork, 0));
  }
  launch_shade_class<SHADE_MISS>(ctx, s[SHADE_MISS], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  launch_shade_class<SHADE_BRDF_DIFFUSE>(ctx, s[SHADE_BRDF_DIFFUSE], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  launch_shade_class<SHADE_BRDF_SPECULAR>(ctx, s[SHADE_BRDF_SPECULAR], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  launch_shade_class<SHADE_BSDF_SPECULAR>(ctx, s[SHADE_BSDF_SPECULAR], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  launch_shade_class<SHADE_BRDF_GGX>(ctx, s[SHADE_BRDF_GGX], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  launch_shade_class<SHADE_BSDF_GGX>(ctx, s[SHADE_BSDF_GGX], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  launch_shade_class<SHADE_OTHER>(ctx, s[SHADE_OTHER], grid, a, sc, bins, binStride, binCounts, qOut, countOut, shadowQueue, shadowCount, tex, deferRR, primary);
  RTC_CUDA(cudaGetLastError());      // a failed launch surfaces here, not in an unrelated later call
  for (int k = 0; k < 6; ++k)
  {
    RTC_CUDA(cudaEventRecord(ctx->shadeJoin[k], ctx->shadeStreams[k]));
    RTC_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->shadeJoin[k], 0));
  }
  return 0;
}

// scratch of the ordered any-hit processing: two queues of `capacity` path ids + {count 0, count 1, cursor, pad}
int ensure_cutout_buffers(rtc_context* ctx, uint64_t capacity)
{
  WavefrontBuffers& wf = ctx->wf;
  if (wf.cutCapacity >= capacity) return 0;
  if (wf.cutBase)
  {
    RTC_CUDA(cudaStreamSynchronize(ctx->stream));
    release_cutout_graph(ctx);         // it captured pointers into this allocation
    RTC_CUDA(cudaFree(wf.cutBase)); wf.cutBase = nullptr; wf.cutCapacity = 0;
  }
  const uint64_t q = (4 * capacity + 255u) & ~(uint64_t)255u;
  void* base = nullptr;
  RTC_CUDA(cudaMalloc(&base, 2 * q + 256));
  char* b = static_cast<char*>(base);
  wf.cutBase = base; wf.cutCapacity = capacity;
  wf.cutQueue[0] = (uint32_t*)b; wf.cutQueue[1] = (uint32_t*)(b + q); wf.cutCounters = (uint32_t*)(b + 2 * q);
  return 0;
}

inline CutoutNext* cutout_next(const WavefrontBuffers& wf) { return reinterpret_cast<CutoutNext*>(wf.cutCounters + 16); }

// ---- the any-hit rounds as a device-side loop -------------------------------------------------------------------------------
// The rounds "play the any-hit program on the closest candidates -> re-trace the ignored ones" repeat until no candidate was
// ignored.  Round 1 reads the depth's own queue and is launched normally; the remaining rounds are a CUDA graph with a
// conditional WHILE node whose body holds two rounds (the ping-pong of the two scratch queues makes every kernel argument
// static) and whose condition is set on the device from the ignored-candidate counter (cudaGraphSetConditional).  No host
// synchronisation: a launch of a scene with cutout materials is as asynchronous as any other.  One graph pair per wavefront
// allocation / scene / SystemData (without iterationIndex, which no captured kernel reads), captured again when one of them
// changes.  The graph is released wherever what it points at is freed (wavefront or scratch regrowth, rtc_scene_destroy), so a
// new allocation or scene that happens to get the old address is never served by a stale capture.
struct CutoutGraph
{
  cudaGraphExec_t radiance = nullptr, shadow = nullptr;
  cudaGraph_t radianceGraph = nullptr, shadowGraph = nullptr;
  const void* wfBase = nullptr; const void* cutBase = nullptr; const void* scene = nullptr;
  rt_SystemData sys{};       // iterationIndex zeroed
  int grid = 0;
};

// Adds the WHILE loop of the any-hit rounds to `graph`; the caller owns the graph (and destroys it when this fails).
int fill_cutout_loop(rtc_context* ctx, const SceneRecord* scene, const WfArgs& a, int grid, bool shadow, cudaGraph_t graph)
{
  const WavefrontBuffers& wf = ctx->wf;
  cudaGraphConditionalHandle handle;
  RTC_CUDA(cudaGraphConditionalHandleCreate(&handle, graph, 0, cudaGraphCondAssignDefault));
  // root: the condition from round 1's counter
  cudaGraphNode_t condKernel = nullptr;
  {
    cudaKernelNodeParams kp{};
    const uint32_t* counter = wf.cutCounters + 0;
    void* args[2] = { &handle, &counter };
    kp.func = (void*)k_cutout_condition; kp.gridDim = dim3(1); kp.blockDim = dim3(1); kp.kernelParams = args;
    RTC_CUDA(cudaGraphAddKernelNode(&condKernel, graph, nullptr, 0, &kp));
  }
  cudaGraphNodeParams wp{};
  wp.type = cudaGraphNodeTypeConditional;
  wp.conditional.handle = handle; wp.conditional.type = cudaGraphCondTypeWhile; wp.conditional.size = 1;
  cudaGraphNode_t whileNode = nullptr;
  RTC_CUDA(cudaGraphAddNode(&whileNode, graph, &condKernel, 1, &wp));
  cudaGraph_t body = wp.conditional.phGraph_out[0];
  // body: two rounds, captured from the ordinary launch code
  const bool wasProfiling = ctx->profiling;
  ctx->profiling = false;                       // event pairs cannot be timed from inside a graph; the caller brackets the whole loop
  const cudaError_t eb = cudaStreamBeginCaptureToGraph(ctx->stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed);
  if (eb != cudaSuccess)
  {
    ctx->profiling = wasProfiling;
    return rtc_set_error(__FILE__, __LINE__, "cudaStreamBeginCaptureToGraph(any-hit rounds)", (int)eb, cudaGetErrorString(eb));
  }
  int rc = 0;
  for (int o = 0; o < 2 && rc == 0; ++o)
  {
    // re-trace the candidates round o ignored, then play the any-hit program on what they found: ignored ones -> queue 1 - o
    const int p = 1 - o;
    if (shadow) rc = launch_connect_closest(ctx, &scene->desc, wf, wf.cutQueue[o], wf.cutCounters + o, wf.cutCounters + 2, true);
    else        rc = launch_extend_after(ctx, &scene->desc, wf, wf.cutQueue[o], wf.cutCounters + o, wf.cutCounters + 2);
    if (rc == 0 && cudaMemsetAsync(wf.cutCounters + p, 0, sizeof(uint32_t), ctx->stream) != cudaSuccess) rc = -1;
    if (rc == 0)
    {
      if (shadow) k_cutout_shadow<<<grid, kBlock, 0, ctx->stream>>>(a, scene->desc, wf.cutQueue[o], wf.cutCounters + o, wf.cutQueue[p], wf.cutCounters + p, cutout_next(wf));
      else        k_cutout_radiance<<<grid, kBlock, 0, ctx->stream>>>(a, scene->desc, wf.cutQueue[o], wf.cutCounters + o, wf.cutQueue[p], wf.cutCounters + p);
    }
  }
  if (rc == 0) k_cutout_condition<<<1, 1, 0, ctx->stream>>>(handle, wf.cutCounters + 0);
  cudaGraph_t captured = nullptr;
  const cudaError_t e = cudaStreamEndCapture(ctx->stream, &captured);
  ctx->profiling = wasProfiling;
  if (rc != 0 || e != cudaSuccess)
  {
    cudaGetLastError();
    if (rc != 0) return rc;
    return rtc_set_error(__FILE__, __LINE__, "cudaStreamEndCapture(any-hit rounds)", (int)e, cudaGetErrorString(e));
  }
  return 0;
}

int build_cutout_loop(rtc_context* ctx, const SceneRecord* scene, const WfArgs& a, int grid, bool shadow, cudaGraph_t* outGraph, cudaGraphExec_t* outExec)
{
  cudaGraph_t graph = nullptr;
  RTC_CUDA(cudaGraphCreate(&graph, 0));
  int rc = fill_cutout_loop(ctx, scene, a, grid, shadow, graph);
  cudaGraphExec_t exec = nullptr;
  if (rc == 0)
  {
    const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
    if (ei != cudaSuccess) rc = rtc_set_error(__FILE__, __LINE__, "cudaGraphInstantiate(any-hit rounds)", (int)ei, cudaGetErrorString(ei));
  }
  if (rc != 0) { cudaGraphDestroy(graph); return rc; }
  *outGraph = graph; *outExec = exec;
  return 0;
}

void destroy_cutout_graph(CutoutGraph* g)
{
  if (!g) return;
  if (g->radiance) cudaGraphExecDestroy(g->radiance);
  if (g->shadow) cudaGraphExecDestroy(g->shadow);
  if (g->radianceGraph) cudaGraphDestroy(g->radianceGraph);
  if (g->shadowGraph) cudaGraphDestroy(g->shadowGraph);
  *g = CutoutGraph();
}

int ensure_cutout_graph(rtc_context* ctx, const SceneRecord* scene, const WfArgs& a, int grid)
{
  CutoutGraph* g = static_cast<CutoutGraph*>(ctx->cutoutGraph);
  if (!g) { g = new CutoutGraph(); ctx->cutoutGraph = g; }
  const WavefrontBuffers& wf = ctx->wf;
  rt_SystemData sys = a.sys;
  sys.iterationIndex = 0;                             // Device::launch writes a new one before every launch
  if (g->radiance && g->wfBase == wf.base && g->cutBase == wf.cutBase && g->scene == scene && g->grid == grid && std::memcmp(&g->sys, &sys, sizeof(rt_SystemData)) == 0)
    return 0;
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));      // an old graph may still be running
  destroy_cutout_graph(g);
  if (int rc = build_cutout_loop(ctx, scene, a, grid, false, &g->radianceGraph, &g->radiance)) { destroy_cutout_graph(g); return rc; }
  if (int rc = build_cutout_loop(ctx, scene, a, grid, true, &g->shadowGraph, &g->shadow)) { destroy_cutout_graph(g); return rc; }
  g->wfBase = wf.base; g->cutBase = wf.cutBase; g->scene = scene; g->grid = grid; g->sys = sys;
  ctx->cutoutGraphBuilds++;
  return 0;
}

// After extend: play __anyhit__radiance_cutout on the closest candidates, re-trace the ignored ones, repeat until none is ignored.
int resolve_radiance_candidates(rtc_context* ctx, const SceneRecord* scene, const WfArgs& a, int grid, const uint32_t* queue, const uint32_t* count)
{
  const WavefrontBuffers& wf = ctx->wf;
  if (int rc = ensure_cutout_graph(ctx, scene, a, grid)) return rc;
  RTC_CUDA(cudaMemsetAsync(wf.cutCounters + 0, 0, sizeof(uint32_t), ctx->stream));
  if (int rc = profile_begin(ctx, RTC_KERNEL_SHADE)) return rc;
  k_cutout_radiance<<<grid, kBlock, 0, ctx->stream>>>(a, scene->desc, queue, count, wf.cutQueue[0], wf.cutCounters + 0);
  if (int rc = profile_end(ctx)) return rc;
  if (int rc = profile_begin(ctx, RTC_KERNEL_EXTEND)) return rc;       // the whole loop (re-traces dominate) as one span
  RTC_CUDA(cudaGraphLaunch(static_cast<CutoutGraph*>(ctx->cutoutGraph)->radiance, ctx->stream));
  ctx->kernelLaunches += 6;                                            // one body execution; further rounds are not counted
  return profile_end(ctx);
}

// Instead of connect: shadow rays as ordered closest-hit queries with __anyhit__shadow / __anyhit__shadow_cutout per candidate.
int resolve_shadow_candidates(rtc_context* ctx, const SceneRecord* scene, const WfArgs& a, int grid, const uint32_t* shadowCount,
                              uint32_t* queueNext, uint32_t* countNext)
{
  const WavefrontBuffers& wf = ctx->wf;
  const uint32_t* queue = wf.shadowQueue; const uint32_t* count = shadowCount;
  k_set_cutout_next<<<1, 1, 0, ctx->stream>>>(cutout_next(wf), queueNext, countNext);
  if (int rc = launch_connect_closest(ctx, &scene->desc, wf, queue, count, wf.cutCounters + 2, false)) return rc;
  if (int rc = ensure_cutout_graph(ctx, scene, a, grid)) return rc;
  RTC_CUDA(cudaMemsetAsync(wf.cutCounters + 0, 0, sizeof(uint32_t), ctx->stream));
  if (int rc = profile_begin(ctx, RTC_KERNEL_SHADE)) return rc;
  k_cutout_shadow<<<grid, kBlock, 0, ctx->stream>>>(a, scene->desc, queue, count, wf.cutQueue[0], wf.cutCounters + 0, cutout_next(wf));
  if (int rc = profile_end(ctx)) return rc;
  if (int rc = profile_begin(ctx, RTC_KERNEL_CONNECT)) return rc;
  RTC_CUDA(cudaGraphLaunch(static_cast<CutoutGraph*>(ctx->cutoutGraph)->shadow, ctx->stream));
  ctx->kernelLaunches += 7;
  return profile_end(ctx);
}

} // namespace

void release_cutout_graph(rtc_context* ctx)
{
  destroy_cutout_graph(static_cast<CutoutGraph*>(ctx->cutoutGraph));
  delete static_cast<CutoutGraph*>(ctx->cutoutGraph);
  ctx->cutoutGraph = nullptr;
}

// ---- schedule tuner (rtc_internal.h ScheduleTuner; the state machine lives in schedule_tuner.h so that a CPU test can run it) ----
namespace {

// With lazy module loading a kernel is loaded at its first launch; the tuner must not time that.
void preload_capped_kernels()
{
  cudaFuncAttributes attr;
  cudaFuncGetAttributes(&attr, k_extend_primary<false, 1>);
  cudaFuncGetAttributes(&attr, k_extend_primary<false, 2>);
  preload_capped_trace_kernels();
  cudaGetLastError();
}

} // namespace

void tuner_finish(rtc_context* ctx) { rtc_tuner::finish(ctx); }
void tuner_release(rtc_context* ctx) { rtc_tuner::release(ctx); }

int launch_wavefront(rtc_context* ctx, const rt_SystemData& sys, uint32_t w, uint32_t h, int raygen, int miss, int iterFirst, int iterCount,
                     int accumFirst, bool countWork)
{
  if (sys.topObject == 0) RTC_FAIL("SystemData.topObject is null (call rtc_ias_build first)");
  const SceneRecord* scene = nullptr;
  for (const SceneRecord* s : ctx->scenes) if ((uint64_t)(uintptr_t)s->d_desc == sys.topObject) scene = s;
  if (!scene) RTC_FAIL("SystemData.topObject was not returned by rtc_ias_build on this context");
  const int maxDepth = sys.pathLengths.y;
  if (maxDepth > 63) RTC_FAIL("pathLengths.y > 63 is not supported");
  const uint64_t pixels = (uint64_t)w * h;
  if (pixels == 0 || iterCount <= 0) return 0;
  // iterations in flight per batch: up to kMaxPathsInFlight paths (deep bounces have few live paths, so the more
  // iterations share a launch the smaller the tail of the persistent traversal kernels); RTC_MAX_PATHS overrides
  uint64_t maxPaths = kMaxPathsInFlight;
  if (const char* env = getenv("RTC_MAX_PATHS")) { const long long v = atoll(env); if (v > 0) maxPaths = (uint64_t)v; }
  uint64_t perBatch = maxPaths / pixels; if (perBatch < 1) perBatch = 1; if (perBatch > (uint64_t)iterCount) perBatch = (uint64_t)iterCount;
  if (pixels * perBatch > 0x7fffffffull) RTC_FAIL("launch too large");
  // 320 B of wavefront state per path: the batch shrinks (down to one iteration) when the device cannot hold it -- other
  // contexts on the same GPU, a smaller GPU, memory held by the caller -- instead of failing the launch
  for (;;)
  {
    bool oom = false;
    const int rc = ensure_wavefront(ctx, pixels * perBatch, &oom);
    if (rc == 0) break;
    if (!oom || perBatch == 1) return rc;
    perBatch = (perBatch + 1) / 2;
  }
  // Material textures (off in every BASELINE configuration, like the reference's GUI default): `cutout` switches to the ordered
  // any-hit processing, whose rounds repeat on the device without a host synchronisation; `tex` selects the texture-aware
  // shade kernels.
  const bool cutout = scene->numCutout > 0;
  const bool tex = cutout || scene->albedoTextures;
  if (cutout) { if (int rc = ensure_cutout_buffers(ctx, pixels * perBatch)) return rc; }

  const int gridShade = ctx->numSMs * 16;     // swept (tools/sweep_shade_block.sh): 8 -> 16 CTAs of 256 per SM in the grid, +0.8 %; the CTA size itself is flat from 128 to 512
  for (int done = 0; done < iterCount; done += (int)perBatch)
  {
    const int batch = (iterCount - done < (int)perBatch) ? iterCount - done : (int)perBatch;
    WfArgs a;
    a.wf = ctx->wf; a.sys = sys; a.launchWidth = w; a.launchHeight = h; a.raygen = raygen; a.miss = miss;
    a.iterFirst = iterFirst + done; a.iterCount = batch; a.accumFirst = accumFirst + done; a.numPaths = (uint32_t)(pixels * (uint64_t)batch);
    // schedule tuner: scenes without cutout materials, timed launches only
    const int tuneSlot = rtc_tuner::begin(ctx, a.numPaths, !countWork && !cutout, preload_capped_kernels);
    uint32_t* cnt = ctx->wf.counters;
    RTC_CUDA(cudaMemsetAsync(cnt, 0, 4 * kNumCounters, ctx->stream));
    // Fused primary path (scenes without material textures): no generate pass.  The depth-0 extend computes its rays from the
    // launch index, and the depth-0 shade kernels recompute the path start instead of reading five state arrays back.
    const bool fused = !tex && 0 < maxDepth;      // pathLengths.y == 0: nothing is traced, generate still zeroes the radiance
    if (!fused)
    {
      if (int rc = profile_begin(ctx, RTC_KERNEL_GENERATE)) return rc;
      k_generate<<<gridShade, kBlock, 0, ctx->stream>>>(a, ctx->wf.queueA, cnt + 0);
      ctx->kernelLaunches++;
      if (int rc = profile_end(ctx)) return rc;
    }
    uint32_t* qIn = ctx->wf.queueA; uint32_t* qOut = ctx->wf.queueB;
    for (int d = 0; d < maxDepth; ++d)
    {
      const bool primary = fused && d == 0;
      if (primary)
      {
        if (int rc = profile_begin(ctx, RTC_KERNEL_EXTEND)) return rc;
        ExtendPrimary policy = { a };
        const int gridTrace = ctx->numSMs * RTC_TRACE_MIN_BLOCKS;
        if (countWork) k_extend_primary<true><<<gridTrace, kPrimaryBlock, 0, ctx->stream>>>(scene->desc, policy, a.numPaths, cnt + 128, ctx->d_launchCounts);
        else if (ctx->traceSchedule == RTC_SCHEDULE_ONE_TRI) k_extend_primary<false, 1><<<gridTrace, kPrimaryBlock, 0, ctx->stream>>>(scene->desc, policy, a.numPaths, cnt + 128, nullptr);
        else if (ctx->traceSchedule == RTC_SCHEDULE_TWO_TRI) k_extend_primary<false, 2><<<gridTrace, kPrimaryBlock, 0, ctx->stream>>>(scene->desc, policy, a.numPaths, cnt + 128, nullptr);
        else           k_extend_primary<false><<<gridTrace, kPrimaryBlock, 0, ctx->stream>>>(scene->desc, policy, a.numPaths, cnt + 128, nullptr);
        ctx->kernelLaunches++;
        RTC_CUDA(cudaGetLastError());
        if (int rc = profile_end(ctx)) return rc;
      }
      else if (int rc = launch_extend(ctx, &scene->desc, ctx->wf, qIn, cnt + d, cnt + 128 + d, countWork)) return rc;
      if (cutout) { if (int rc = resolve_radiance_candidates(ctx, scene, a, gridShade, qIn, cnt + d)) return rc; }
      if (int rc = profile_begin(ctx, RTC_KERNEL_SHADE)) return rc;
      uint32_t* binCounts = cnt + 256 + d * 8;
      k_bin<<<gridShade, kBlock, 0, ctx->stream>>>(a, scene->desc, primary ? nullptr : qIn, cnt + d, ctx->wf.bins, ctx->wf.binStride, binCounts, cnt + d);
      if (int rc = launch_shade_classes(ctx, gridShade, a, scene->desc, ctx->wf.bins, ctx->wf.binStride, binCounts, qOut, cnt + d + 1, ctx->wf.shadowQueue, cnt + 64 + d, tex, cutout, primary)) return rc;
      ctx->kernelLaunches += 1 + SHADE_NUM_CLASSES;
      if (int rc = profile_end(ctx)) return rc;
      if (sys.numLights > 0)
      {
        if (cutout) { if (int rc = resolve_shadow_candidates(ctx, scene, a, gridShade, cnt + 64 + d, qOut, cnt + d + 1)) return rc; }
        else        { if (int rc = launch_connect(ctx, &scene->desc, ctx->wf, cnt + 64 + d, cnt + 192 + d, countWork)) return rc; }
      }
      uint32_t* t = qIn; qIn = qOut; qOut = t;
    }
    if (int rc = profile_begin(ctx, RTC_KERNEL_ACCUMULATE)) return rc;
    k_accumulate<<<(unsigned)((pixels + kBlock - 1) / kBlock), kBlock, 0, ctx->stream>>>(a);
    if (int rc = profile_end(ctx)) return rc;
    k_stats<<<1, 32, 0, ctx->stream>>>(cnt, maxDepth, a.numPaths, ctx->d_stats);
    ctx->kernelLaunches += 2;
    RTC_CUDA(cudaGetLastError());
    rtc_tuner::end(ctx, tuneSlot);
  }
  return 0;
}

int read_stack_overflows_primary(rtc_context* ctx, uint64_t* out)
{
  unsigned int v = 0;
  RTC_CUDA(cudaMemcpyFromSymbolAsync(&v, g_rtcStackOverflowsPrimary, sizeof(v), 0, cudaMemcpyDeviceToHost, ctx->stream));
  RTC_CUDA(cudaStreamSynchronize(ctx->stream));
  *out = v;
  return 0;
}

int launch_generate_primary(rtc_context* ctx, const rt_SystemData& sys, uint32_t w, uint32_t h, int iteration, rtc_ray* rays)
{
  const uint64_t n = (uint64_t)w * h;
  if (n == 0) return 0;
  k_generate_primary<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, ctx->stream>>>(sys, w, h, iteration, reinterpret_cast<float4*>(rays));
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

int launch_composite(rtc_context* ctx, const rt_CompositorData& args)
{
  if (args.launchWidth <= 0 || args.resolution.y <= 0) return 0;
  dim3 grid((unsigned)((args.launchWidth + kBlock - 1) / kBlock), (unsigned)args.resolution.y);
  k_composite<<<grid, kBlock, 0, ctx->stream>>>(args);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

int launch_tonemap(rtc_context* ctx, const rt_TonemapperParams& p, const float4* rgba, uint8_t* rgb, uint64_t n)
{
  if (n == 0) return 0;
  k_tonemap<<<(unsigned)((n + kBlock - 1) / kBlock), kBlock, 0, ctx->stream>>>(p, rgba, rgb, n);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Test hook (rtc_probe_math): the arithmetic the shading kernels are DEFINED by -- the pinned transcendentals of
// include/rt_portable_math.h plus IEEE division and square root -- evaluated element-wise with exactly this translation
// unit's compiler flags (-fmad=false -prec-div=true -prec-sqrt=true).  tests/test_gpu_edge_cases.py compares the bits with
// the same header compiled by gcc, input by input, instead of only through rendered frames.
namespace {
__global__ void __launch_bounds__(kBlock)
k_probe_math(int fn, const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ out, uint32_t n)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float a = x[i], b = y[i];
  float r;
  switch (fn)
  {
    case RTC_MATH_SIN:   r = rt_sinf(a); break;
    case RTC_MATH_COS:   r = rt_cosf(a); break;
    case RTC_MATH_ATAN:  r = rt_atanf(a); break;
    case RTC_MATH_ATAN2: r = rt_atan2f(a, b); break;
    case RTC_MATH_ACOS:  r = rt_acosf(a); break;
    case RTC_MATH_EXP:   r = rt_expf(a); break;
    case RTC_MATH_LOG:   r = rt_logf(a); break;
    case RTC_MATH_POW:   r = rt_powf(a, b); break;
    case RTC_MATH_DIV:   r = a / b; break;
    case RTC_MATH_SQRT:  r = sqrtf(a); break;
    case RTC_MATH_MULADD: r = a * b + a; break;        // must stay two roundings (no contraction)
    default:             r = 0.0f; break;
  }
  out[i] = r;
}
} // namespace

int launch_probe_math(rtc_context* ctx, int fn, const float* x, const float* y, float* out, uint32_t n)
{
  if (n == 0) return 0;
  k_probe_math<<<(n + kBlock - 1) / kBlock, kBlock, 0, ctx->stream>>>(fn, x, y, out, n);
  ctx->kernelLaunches++;
  RTC_CUDA(cudaGetLastError());
  return 0;
}
