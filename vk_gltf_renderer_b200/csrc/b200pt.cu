// b200pt.cu — wavefront path-tracer kernels for sm_100a + the C-ABI of include/b200pt.h.
//
// Stage map (reference function -> kernel), SURVEY.md Appendix C:
//   processPixel head / samplePixel / getRay      gltf_pathtrace.slang:546-581,502-530  -> k_raygen (+ regen in finalizeSample)
//   IRaytracer::Trace: tree walks                  raytracer_interface.h.slang:69-122    -> k_trace (persistent warps)
//                      any-hit alpha tests         raytracer_interface.h.slang:82-112    -> k_alpha<false> (dense)
//   pathTraceOneBounce                             gltf_pathtrace.slang:87-430           -> k_shade
//   IRaytracer::TraceShadow: tree walks            raytracer_interface.h.slang:139-187   -> k_shadow (persistent warps)
//                      any-hit transmission        raytracer_interface.h.slang:149-179   -> k_alpha<true> (dense)
//   NEE add + RR + depth++ (pathTrace tail)        gltf_pathtrace.slang:462-485          -> k_resolve
//   accumulation                                   gltf_pathtrace.slang:582-630          -> k_accumulate
//   shadow catcher (handleShadowCatcher)           pathtrace_functions.h.slang:499-554   -> k_shade (light sample) + shadow kernels + finishPost
//   eOptixAlbedoNormal guide image                 gltf_pathtrace.slang:240-263,653-670  -> capture in k_shade, k_guide
// Next to the frame path (SURVEY.md section 8 f):
//   morph.comp / skinning.comp                     shaders/*.comp.slang                  -> k_morph, k_skin, k_regather_shade (animate.cuh)
//   world_matrix_propagate / update_render_instances                                     -> k_propagate_level, k_update_render_nodes
//   BLAS / TLAS build and update                   src/gltf_scene_rtx.cpp:173-503        -> k_lbvh_* (lbvh.cuh), k_refit_* (refit.cuh)
//   GltfRenderer::tonemap                          src/renderer.cpp:992-1054             -> k_tm_histogram, k_tm_exposure, k_tonemap (tonemap.cuh)
// One path slot per pixel; samples of a pixel within a frame run back to back in the same slot
// (path regeneration) because the reference continues ONE rng stream across a pixel's samples.
#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "bvh.h"
#include "animate.cuh"
#include "lbvh.cuh"
#include "shade.cuh"
#include "tonemap.cuh"

using namespace pt;

static_assert(sizeof(b200pt_render_node) == 136, "GltfRenderNode layout");
static_assert(sizeof(b200pt_texture_info) == 32, "GltfTextureInfo layout");
static_assert(sizeof(b200pt_shade_material) == 288, "GltfShadeMaterial layout");
static_assert(sizeof(b200pt_light) == 64, "GltfLight layout");
static_assert(sizeof(b200pt_frame_info) == 396, "SceneFrameInfo layout");
static_assert(sizeof(b200pt_push_constant) == 48, "PathtracePushConstant layout");

namespace {

constexpr int kMaxIters = 4096;  // per-frame iteration counter slots
// Any-hit continuation rounds per bounce: a ray whose kCand candidates were all rejected goes through another k_trace / k_shadow round
// that resumes behind the last one; after kContRounds rounds whatever is still undecided finishes inside the last k_alpha.  Measured on
// the bench scene (r02zg / r02zh, one box each): 4 candidates x 1 round 984 / 977 Mray/s -- the in-kernel fallback walks of the last
// k_alpha (2 of 32 lanes busy) were a tail on every bounce -- x 2 rounds 1019.8 / 1022.8, x 3 / 4 / 6 rounds 1011 / 1016 / 1014;
// 2 candidates (the bound shrinks sooner) x 2 / 3 / 4 / 5 / 6 / 8 rounds 987 / 1012 / 1024 + 1022 / 1016 / 1020 / 1014: the same
// plateau with more launches.  Counter arrays per lane: 5 (trace / post queues and cursors, shadow queue) + per ray kind
// (rounds + 1) any-hit counters, rounds continuation counters and rounds continuation cursors.
constexpr int kContRounds = 2;
constexpr int kCounterArrays = 5 + 2 * (3 * kContRounds + 1);

// -------------------------------------------------------------------------------------------------
// queue helper: warp-aggregated append
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void queuePush(uint32_t* q, uint32_t* cnt, uint32_t value)
{
  const unsigned mask = __activemask();
  const int      lane = threadIdx.x & 31;
  const int      leader = __ffs(mask) - 1;
  uint32_t       base = 0;
  if(lane == leader)
    base = atomicAdd(cnt, (uint32_t)__popc(mask));
  base = __shfl_sync(mask, base, leader);
  q[base + __popc(mask & ((1u << lane) - 1u))] = value;
}

__device__ __forceinline__ void statAdd(unsigned long long* p, unsigned long long v)
{
  // per-warp aggregation of a uniform +v
  const unsigned mask = __activemask();
  const int      lane = threadIdx.x & 31;
  if(lane == __ffs(mask) - 1)
    atomicAdd(p, v * (unsigned long long)__popc(mask));
}

// -------------------------------------------------------------------------------------------------
// camera ray + sample start (samplePixel head: gltf_pathtrace.slang:502-530; getRay: pathtrace_functions.h.slang:791-811)
// -------------------------------------------------------------------------------------------------
__device__ void startSample(const PathState& P, const FrameParams& F, uint32_t i, uint32_t seed, float2 jitter, uint32_t sampleIdx)
{
  const uint32_t px = pixelOf(F, i);
  const uint32_t x = px % (uint32_t)F.width;
  const uint32_t y = pixelRow(F, px);
  const Mat4&    projI = *reinterpret_cast<const Mat4*>(F.fi.projInv);
  const Mat4&    viewI = *reinterpret_cast<const Mat4*>(F.fi.viewInv);
  const bool     ortho = (F.fi.flags & B200PT_SCENE_IS_ORTHOGRAPHIC) != 0;
  const float2   clip = f2(((float)x + jitter.x) / F.fi.imageSize[0] * 2.0f - 1.0f, ((float)y + jitter.y) / F.fi.imageSize[1] * 2.0f - 1.0f);
  float4         vc = mul_vM(f4(clip.x, clip.y, -1.0f, 1.0f), projI);
  vc = vc / vc.w;
  float3 org, dir;
  if(ortho)
  {
    org = xyz(mul_vM(vc, viewI));
    dir = normalize(xyz(mul_vM(f4(0, 0, -1, 0), viewI)));
  }
  else
  {
    org = f3(viewI.m[12], viewI.m[13], viewI.m[14]);
    dir = normalize(xyz(mul_vM(vc, viewI)) - org);
    // thin-lens DOF: the two rand() are consumed even when aperture == 0 (:519-520)
    const float3 focalPoint = dir * F.pc.focalDistance;
    const float  cam_r1 = rnd(seed) * kTwoPi;
    const float  cam_r2 = rnd(seed) * F.pc.aperture;
    const float4 camRight = mul_Mv(viewI, f4(1, 0, 0, 0));
    const float4 camUp = mul_Mv(viewI, f4(0, 1, 0, 0));
    const float3 rap = (xyz(camRight) * cosf(cam_r1) + xyz(camUp) * sinf(cam_r1)) * sqrtf(cam_r2);
    dir = normalize(focalPoint - rap);
    org += rap;
  }
  dir = normalize(dir);  // pathTrace() re-normalises at the top of every loop iteration (:447)
  P.rayO[i] = f4(org, 0.0f);
  P.rayD[i] = f4(dir, kInfinite);
  P.thr[i] = f4(1.0f, 1.0f, 1.0f, kDirac);
  P.rad[i] = f4(0.0f, 0.0f, 0.0f, __uint_as_float(0u));
  P.misc[i] = f4(0.0f, 0.0f, __uint_as_float(PF_SOLID), __uint_as_float(seed));
  P.medium[i] = make_uint4(0u, 0u, 0u, sampleIdx << 16);
  if(isFirstFrame(F, i))
    P.firstHit[i] = f4(1e34f, 1e34f, 1e34f, 1.0f);  // PathTracerState::firstHitPos sentinel, pt.solid = true
  if(P.guideA)
  {
    P.guideA[i] = f4(0.f, 0.f, 0.f, 0.f);  // GuideScratch defaults: albedo 0, normalRoughness 0
    P.guideN[i] = f4(0.f, 0.f, 0.f, 0.f);
  }
}

// end of one samplePixel(): firefly clamp, add to the pixel sum, start the pixel's next sample if any
__device__ void finalizeSample(const PathState& P, const FrameParams& F, uint32_t i, float3 radiance, bool solid, uint32_t seed, uint32_t sampleIdx,
                               uint32_t* qNext, uint32_t* cntNext, DevStats* stats)
{
  float4      r = f4(radiance, solid ? 1.0f : 0.0f);
  const float lum = (r.x + r.y + r.z) * (1.0f / 3.0f);
  if(lum > F.pc.fireflyClampThreshold)
    r = r * (F.pc.fireflyClampThreshold / lum);
  P.pixSum[i] = P.pixSum[i] + r;
  const uint32_t s = sampleIdx + 1;
  if((int)s < F.pc.numSamples)
  {
    const float a = rnd(seed), b = rnd(seed);
    startSample(P, F, i, seed, f2(a, b), s);
    statAdd(&stats->pathsStarted, 1ull);
    queuePush(qNext, cntNext, i);
  }
}

// -------------------------------------------------------------------------------------------------
// kernels
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_raygen(PathState P, const __grid_constant__ FrameParams F, uint32_t* qTrace, uint32_t* cnt0, DevStats* stats)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < F.numPaths; i += stride)
  {
    const uint32_t px = pixelOf(F, i);
    const uint32_t x = px % (uint32_t)F.width;
    const uint32_t y = pixelRow(F, px);
    uint32_t       seed = xxhash32(x, y, (uint32_t)F.pc.frameCount + frameOf(F, i));
    const float    u1 = rnd(seed), u2 = rnd(seed);
    // sampleGaussian (pathtrace_functions.h.slang:784-789), sigma = 0.4246609 px
    const float  rr = sqrtf(-2.0f * logf(fmaxf(1e-38f, u1)));
    const float  theta = 2.0f * kPi * u2;
    const float2 jitter = f2(0.5f + (rr * cosf(theta)) * 0.4246609f, 0.5f + (rr * sinf(theta)) * 0.4246609f);
    P.pixSum[i] = f4(0.f, 0.f, 0.f, 0.f);
    startSample(P, F, i, seed, jitter, 0u);
    qTrace[i] = i;
  }
  if(blockIdx.x == 0 && threadIdx.x == 0)
  {
    *cnt0 = F.numPaths;
    atomicAdd(&stats->pathsStarted, (unsigned long long)F.numPaths);
  }
}

// Persistent-warp scheme (Aila & Laine 2009 style): all 32 lanes of a warp reconverge at the fetch point
// (__syncwarp), lanes that finished their ray take the next queue entries from a global cursor, then the
// warp walks the tree until fewer than kRefillThreshold lanes are still busy and goes back to refill.
constexpr int kRefillThreshold = 22;
// a lane's pending triangle group is postponed while fewer than 1 / 2^kPostponeShift of the warp's lanes have one (TravState::step)
constexpr int kPostponeShift = 2;

// full-warp fetch: every lane calls it; lanes with need==true receive the next queue slot or 0xFFFFFFFF
__device__ __forceinline__ uint32_t fetchWork(bool need, uint32_t* workCounter, uint32_t count)
{
  const unsigned want = __ballot_sync(0xffffffffu, need);
  if(want == 0)
    return 0xFFFFFFFFu;
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(want) - 1;
  uint32_t  base = 0;
  if(lane == leader)
    base = atomicAdd(workCounter, (uint32_t)__popc(want));
  base = __shfl_sync(0xffffffffu, base, leader);
  if(!need)
    return 0xFFFFFFFFu;
  const uint32_t k = base + (uint32_t)__popc(want & ((1u << lane) - 1u));
  return k < count ? k : 0xFFFFFFFFu;
}

// IRaytracer::Trace, geometry part, for every path in the queue: ONE walk of the scene tree gives the closest
// FORCE_OPAQUE hit and the kCand nearest any-hit candidates in front of it (traverse.cuh).  The stochastic alpha
// tests need textures and touch only the few lanes whose walk just ended -- inside this kernel they ran with ~2 of
// 32 lanes active and took 17 % of its instructions / 26 % of its stall samples (ncu, profiles/) -- so they live in
// the dense kernel k_alpha; this kernel only writes the candidates out.
// Per lane: path (-1 needs work, -2 exhausted) and a resumable traversal; finished lanes are handled in the
// converged part of the loop, never inside the traversal loop.
// mode: TRACE_CONT = continuation round (the paths in the queue had all kCand candidates rejected by k_alpha and resume
// behind the last one; P.hit seeds the opaque bound and is refined), TRACE_TMIN = rayO.w carries tmin (ray-level API).
constexpr int kTraceMinBlocks = 8;  // 64 registers, no spills: 8 blocks/SM.  Measured: 6 blocks / 80 registers 944, 7 / 72 967 (r02o), 8 / 64 973 (r02q) and 990.8 vs 984.1 (r02x, same box, leaf cost 0.6)
enum : int
{
  TRACE_CONT = 1,
  TRACE_TMIN = 2,
};
template <bool OMM>
__global__ void __launch_bounds__(128, kTraceMinBlocks) k_trace(PathState P, DevScene S, const uint32_t* __restrict__ q, const uint32_t* __restrict__ cntIn,
                                                                       uint32_t* workCounter, uint32_t* qAlpha, uint32_t* cntAlpha, DevStats* stats, int refillThreshold,
                                                                       int postponeShift, int mode)
{
  __shared__ Cand s_cand[kCand * 128];  // candidate lists, one column per thread (20-byte stride: conflict-free)
  Cand* const     cand = &s_cand[threadIdx.x];
  constexpr int   cs = 128;
  const bool      cont = (mode & TRACE_CONT) != 0;
  const uint32_t  count = *cntIn;
  TravState       T;
  uint2           stack[TravState::kStackSize];
  int             path = -1;
  bool            travDone = false;  // traversal finished, write-out pending
  for(;;)
  {
    __syncwarp();
    if(path >= 0 && travDone)
    {
      travDone = false;
      T.flushCounters(&stats->nodesVisited, &stats->trisTested);
      const TraceHit ho = T.result();
      P.hit[path] = f4(ho.t, ho.u, ho.v, __uint_as_float(ho.slot));
      const int n = T.candidatesInFront(cand, cs);
      if(n > 0)
      {
#pragma unroll
        for(int i = 0; i < kCand; i++)
          if(i < n)
          {
            const Cand c = cand[i * cs];
            P.cand[i][path] = f4(c.t, c.u, c.v, __uint_as_float(c.slot));
          }
        P.candInfo[path] = make_uint2((uint32_t)n, cand[(n - 1) * cs].gid);
        queuePush(qAlpha, cntAlpha, (uint32_t)path);
      }
      if(T.overflow)
        atomicOr(&stats->errorFlags, 1ull);
      path = -1;
    }
    __syncwarp();
    // ---- refill ----
    {
      const bool     need = (path == -1);
      const uint32_t k = fetchWork(need, workCounter, count);
      if(need)
      {
        if(k == 0xFFFFFFFFu)
          path = -2;
        else
        {
          path = (int)q[k];
          const float4 o = P.rayO[path];
          const float4 d = P.rayD[path];
          const float  tmin = (mode & TRACE_TMIN) ? o.w : 0.0f;
          if(!cont)
            T.init(S.bvh, xyz(o), xyz(d), tmin, d.w, true, false, false, 0.f, 0u);
          else
          {
            T.init(S.bvh, xyz(o), xyz(d), tmin, d.w, true, false, true, P.cand[kCand - 1][path].x, P.candInfo[path].y);
            const float4 hp = P.hit[path];
            if(__float_as_uint(hp.w) != 0xFFFFFFFFu)
              T.seedOpaque(hp.x, hp.y, hp.z, __float_as_uint(hp.w));
          }
        }
      }
    }
    if(__all_sync(0xffffffffu, path == -2))
      break;
    // ---- traverse: warp-uniform loop (all 32 lanes iterate, idle lanes are predicated off) until too few
    //      lanes are still busy ----
    for(;;)
    {
#ifdef B200PT_COUNT_TRAVERSAL
      {
        const unsigned busy = __ballot_sync(0xffffffffu, path >= 0 && !travDone);
        if((threadIdx.x & 31) == 0)
        {
          atomicAdd(&stats->warpIters, 1ull);
          atomicAdd(&stats->busyLaneIters, (unsigned long long)__popc(busy));
        }
      }
#endif
      if(path >= 0 && !travDone)
        travDone = T.step<kCand, false, OMM, 1>(stack, postponeShift, cand, cs, S.bvh.ommRef, S.bvh.ommData);
      if(__popc(__ballot_sync(0xffffffffu, path >= 0 && !travDone)) < refillThreshold)
        break;
    }
  }
  if(blockIdx.x == 0 && threadIdx.x == 0 && !cont)
    atomicAdd(&stats->closestRays, (unsigned long long)count);
}

// Any-hit part of IRaytracer::Trace (SHADOW = false) and IRaytracer::TraceShadow (SHADOW = true): the candidates
// the geometry kernel collected, nearest first, one rand() each (raytracer_interface.h.slang:82-112, 149-179, with
// the order pinned to (t, triangle id)).
//   Trace:       the first candidate that passes its alpha test replaces the opaque hit.
//   TraceShadow: every candidate that passes multiplies the transmission (0 for MASK / opaque-ish materials);
//                the result is folded into the path's pending NEE contribution.
// kCand lanes per path: lane j evaluates the opacity of candidate j (the texture fetches -- the long latency chain
// -- run in parallel), then all of them replay the same sequential decisions and lane 0 writes.  A path whose
// kCand candidates are used up goes to the continuation queue (another k_trace / k_shadow round resumes the walk
// behind the last candidate); in the last round (qCont == nullptr) it keeps walking right here instead.
template <bool SHADOW>
__global__ void __launch_bounds__(128) k_alpha(PathState P, DevScene S, const uint32_t* __restrict__ q, const uint32_t* __restrict__ cntIn, uint32_t* qCont,
                                               uint32_t* cntCont, DevStats* stats, int mode)
{
  static_assert(kCand == 2 || kCand == 4 || kCand == 8, "kCand lanes per path");
  // candidate slots index the triangle array of the tree that produced them: the merged tree for closest-hit rays,
  // the split opaque / non-opaque arrays for shadow rays
  const uint2* __restrict__ triMeta = SHADOW ? S.triMetaS : S.triMeta;
  constexpr int             KF = 16;  // candidates per walk of the in-kernel fallback (its list lives in local memory)
  stageSrgbLut(S.lutSrgb);
  const uint32_t count = *cntIn;
  constexpr int  G = kCand, PPW = 32 / kCand;  // lanes per path, paths per warp
  const int      lane = threadIdx.x & 31, sub = lane % G, grp = lane / G, base = lane - sub;
  const uint32_t warpsTotal = gridDim.x * (blockDim.x >> 5);
  const uint32_t warpId = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for(uint32_t k0 = warpId * (uint32_t)PPW; k0 < count; k0 += warpsTotal * (uint32_t)PPW)  // warp-uniform trip count
  {
    const uint32_t k = k0 + (uint32_t)grp;
    const bool     valid = k < count;
    uint32_t       path = 0;
    uint2          info = make_uint2(0u, 0u);
    if(valid)
    {
      path = q[k];
      info = P.candInfo[path];
    }
    const int n = (int)(info.x & 0xffu);
    // ---- lane j: candidate j and its opacity ----
    float    ct = 0.f, cu = 0.f, cv = 0.f, op = 0.f, transmission = 0.f;
    uint32_t slot = 0;
    if(sub < n)
    {
      const float4 c = P.cand[sub][path];
      slot = __float_as_uint(c.w);
      // the triangle's pre-gathered alpha record: candidate -> (index ->) record -> texels
      const uint32_t ri = SHADOW ? slot - S.alphaBaseS : __ldg(&S.alphaIdx[slot]);
      const uint32_t w0 = __float_as_uint(__ldg(&(SHADOW ? S.bvhA.tris : S.bvh.tris)[slot * 3 + 0]).w);
      const bool     flip = ((w0 >> 28) & TRI_FLIPPED) != 0;  // mirrored instance: (u, v) swap back
      const AlphaRec rec = loadAlphaRec(S.alphaRecs + ri);
      ct = c.x;
      cu = flip ? c.z : c.y;
      cv = flip ? c.y : c.z;
      op = opacityFromRecord(rec, f3(1.0f - cu - cv, cu, cv));
      transmission = rec.transmission;
    }
    const uint32_t seedIn = valid ? __float_as_uint(P.misc[path].w) : 0u;
    uint32_t       seed = seedIn;
    if(!SHADOW)
    {
      int acc = -1;
#pragma unroll
      for(int i = 0; i < kCand; i++)
      {
        const float oi = __shfl_sync(0xffffffffu, op, base + i);
        if(i < n && acc < 0 && rnd(seed) <= oi)
          acc = i;
      }
      if(acc >= 0 && sub == acc)
        P.hit[path] = f4(ct, cu, cv, __uint_as_float(slot));
      const float    lastT = __shfl_sync(0xffffffffu, ct, base + kCand - 1);
      if(acc < 0 && n == kCand && qCont != nullptr)
      {
        if(sub == 0)
          queuePush(qCont, cntCont, path);
      }
      else if(acc < 0 && n == kCand)
      {
        // every collected candidate was rejected and there may be more: keep walking, kCand at a time (the lanes of
        // the group do this redundantly, lane 0 writes).  Each walk also refines the opaque hit (traverse.cuh).
        const float4 o = P.rayO[path], d = P.rayD[path], hp = P.hit[path];
        const float  tmin = (mode & TRACE_TMIN) ? o.w : 0.0f;
        TraceHit     opq;
        opq.slot = 0xFFFFFFFFu;
        if(__float_as_uint(hp.w) != 0xFFFFFFFFu)
          opq = seedHit(S.bvh, hp.x, hp.y, hp.z, __float_as_uint(hp.w));
        float    loT = lastT;
        uint32_t loId = info.y;
        Cand     cand[KF];
        bool     accepted = false, overflowed = false;
        for(;;)
        {
          const int m = walkCollect<KF>(S.bvh, xyz(o), xyz(d), tmin, d.w, true, false, true, true, loT, loId, opq, cand, &overflowed);
          for(int i = 0; i < m && !accepted; i++)
          {
            const uint2               meta = triMeta[cand[i].slot];
            const bool                flip = ((meta.x >> 28) & TRI_FLIPPED) != 0;
            const float               u = flip ? cand[i].v : cand[i].u, v = flip ? cand[i].u : cand[i].v;
            const b200pt_render_node& node = S.nodes[meta.x & 0x0fffffffu];
            const float               opacity = getOpacity(S, node, S.prims[node.renderPrimID], meta.y, f3(1.0f - u - v, u, v));
            if(rnd(seed) <= opacity)
            {
              if(sub == 0)
                P.hit[path] = f4(cand[i].t, u, v, __uint_as_float(cand[i].slot));
              accepted = true;
            }
          }
          if(accepted || m < KF)
            break;
          loT = cand[KF - 1].t;
          loId = cand[KF - 1].gid;
        }
        if(!accepted && sub == 0 && opq.slot != 0xFFFFFFFFu)
        {
          const TraceHit ho = unflipHit(opq);
          P.hit[path] = f4(ho.t, ho.u, ho.v, __uint_as_float(ho.slot));
        }
        if(overflowed && sub == 0)
          atomicOr(&stats->errorFlags, 1ull);
      }
    }
    else
    {
      // a continuation round resumes with the running transmission and segment start the previous round parked
      // in P.hit (free between shading and the next k_trace)
      const float4 saved = (valid && (mode & TRACE_CONT)) ? P.hit[path] : f4(1.0f, 1.0f, 1.0f, 0.0f);
      float3       total = xyz(saved);
      float        prevHitT = saved.w;
      bool         done = false, parked = false;
      const float4 misc = valid ? P.misc[path] : f4(0, 0, 0, 0);
      bool         isInside = (__float_as_uint(misc.z) & PF_SHADOW_INSIDE) != 0;
      const float3 dir = valid ? xyz(P.shD[path]) : f3(0, 0, 1);
      auto         accept = [&](uint32_t sl, float t, float u, float v) {
        const uint2               meta = triMeta[sl];
        const b200pt_render_node& node = S.nodes[meta.x & 0x0fffffffu];
        const float               seg = fmaxf(0.0f, t - prevHitT);
        const float3              cur = getShadowTransmission(S, node, S.prims[node.renderPrimID], meta.y, f3(1.0f - u - v, u, v), seg, dir, isInside);
        prevHitT = t;
        total *= cur;
        if(maxc(total) <= 0.01f)
        {
          total = f3(0.0f);
          done = true;
        }
      };
#pragma unroll
      for(int i = 0; i < kCand; i++)
      {
        const float    oi = __shfl_sync(0xffffffffu, op, base + i);
        const float    ti = __shfl_sync(0xffffffffu, ct, base + i);
        const float    ui = __shfl_sync(0xffffffffu, cu, base + i);
        const float    vi = __shfl_sync(0xffffffffu, cv, base + i);
        const uint32_t si = __shfl_sync(0xffffffffu, slot, base + i);
        const float    tr = __shfl_sync(0xffffffffu, transmission, base + i);
        if(i < n && !done && rnd(seed) < oi)
        {
          if(tr <= 0.01f)
          {
            // getShadowTransmission returns 0 for a non-transmissive material (alpha-tested foliage): the ray is blocked
            // (same result as accept(), without its gathers)
            prevHitT = ti;
            total = f3(0.0f);
            done = true;
          }
          else
            accept(si, ti, ui, vi);
        }
      }
      const float lastT = __shfl_sync(0xffffffffu, ct, base + kCand - 1);
      if(!done && n == kCand && qCont != nullptr)
      {
        parked = true;
        if(sub == 0)
        {
          P.hit[path] = f4(total, prevHitT);
          const uint32_t fl = (__float_as_uint(misc.z) & ~PF_SHADOW_INSIDE) | (isInside ? PF_SHADOW_INSIDE : 0u);
          reinterpret_cast<uint32_t*>(&P.misc[path])[2] = fl;
          queuePush(qCont, cntCont, path);
        }
      }
      else if(!done && n == kCand)
      {
        // more than kCand layers on the segment: keep walking, kCand at a time (rare)
        const float4 so = P.shO[path];
        float        loT = lastT;
        uint32_t     loId = info.y;
        Cand         cand[KF];
        bool         overflowed = false;
        while(!done)
        {
          TraceHit opq;
          opq.slot = 0xFFFFFFFFu;
          const int m = walkCollect<KF>(S.bvhA, xyz(so), dir, 0.0f, so.w, false, true, true, true, loT, loId, opq, cand, &overflowed);
          if(opq.slot != 0xFFFFFFFFu)
          {
            // (the first walk of the segment found no opaque occluder, so none can turn up here)
            total = f3(0.0f);
            done = true;
          }
          for(int i = 0; i < m && !done; i++)
          {
            const uint2               meta = triMeta[cand[i].slot];
            const bool                flip = ((meta.x >> 28) & TRI_FLIPPED) != 0;
            const float               u = flip ? cand[i].v : cand[i].u, v = flip ? cand[i].u : cand[i].v;
            const b200pt_render_node& node = S.nodes[meta.x & 0x0fffffffu];
            const float               opacity = getOpacity(S, node, S.prims[node.renderPrimID], meta.y, f3(1.0f - u - v, u, v));
            if(rnd(seed) < opacity)
              accept(cand[i].slot, cand[i].t, u, v);
          }
          if(m < KF)
            break;
          loT = cand[KF - 1].t;
          loId = cand[KF - 1].gid;
        }
        if(overflowed && sub == 0)
          atomicOr(&stats->errorFlags, 1ull);
      }
      if(valid && sub == 0 && !parked)
      {
        const float4 c = P.shC[path];
        P.shC[path] = f4(xyz(c) * total, c.w);
      }
    }
    if(valid && sub == 0 && seed != seedIn)
      reinterpret_cast<uint32_t*>(&P.misc[path])[3] = seed;
  }
}

constexpr int kShadeBlock = 512;    // measured: 128 -> 0.50 ms/launch, 256 + barrier 0.41, 512 no barrier 0.475, 512 + barrier 0.33
constexpr int kShadeMinBlocks = 4;  // measured on B200: 3 -> 1.165 ms, 4 -> 1.017, 5 -> 1.029, 6 -> 1.064 per launch
// one barrier per pass; barriers between the four sections of a pass as well were measured: no further gain
template <uint32_t FEAT>
__global__ void __launch_bounds__(kShadeBlock, kShadeMinBlocks * 128 / kShadeBlock) k_shade(PathState P, DevScene S, const __grid_constant__ FrameParams F, const uint32_t* __restrict__ q,
                                               const uint32_t* __restrict__ cntIn, uint32_t* qPost, uint32_t* cntPost, uint32_t* qShadow, uint32_t* cntShadow,
                                                                 uint32_t* qNext, uint32_t* cntNext, DevStats* stats)
{
  stageSrgbLut(S.lutSrgb);
  const uint32_t count = *cntIn;
  const uint32_t stride = gridDim.x * blockDim.x;
  // One path per thread per pass.  The kernel is ~12 000 straight-line instructions that every warp walks once per
  // path, so it is bound by instruction fetch (ncu: no_instruction is its top stall, 20 % issue utilisation); the
  // block-uniform loop with a barrier per pass keeps the warps of a block -- and with kShadeBlock = 512 all four
  // warps of a scheduler -- inside the same stretch of code so they share the fetched lines.
  // pass state shared by the four sections of a pass
  uint32_t                  i = 0, flags = 0, seed = 0, scatterBounces = 0, sampleIdx = 0, depth = 0, slot = 0;
  float4                    hr, misc;
  uint4                     med;
  float3                    org, dir, throughput, radiance;
  float                     coneWidth = 0.f, lastSamplePdf = 0.f, hitT = 0.f, worldFoot = 0.f;
  uint2                     meta;
  const b200pt_render_node* nodeP = nullptr;
  HitState                  hit;
  PbrMaterial               pbrMat;
  DirectLight               directLight;
  bool                      nextEventValid = false;
  bool                      onPlane = false;  // the ray met the infinite ground plane in front of the geometry
  bool                      catcher = false;  // ... and the plane is a shadow catcher (handleShadowCatcher, pathtrace_functions.h.slang:499-554)
#ifdef B200PT_DEBUG
  bool dbgPixel = false;
#endif
  // ---- section 1: path state, environment hit (path ends), hit attributes ----
  auto shadeLoad = [&](const uint32_t k) -> bool {
    i = q[k];
    const float4   ro = P.rayO[i];
    const float4   rd = P.rayD[i];
    hr = P.hit[i];
    float4         thr4 = P.thr[i];
    float4         rad4 = P.rad[i];
    misc = P.misc[i];
    med = P.medium[i];
    org = xyz(ro);
    dir = xyz(rd);
    coneWidth = ro.w;
    throughput = xyz(thr4);
    radiance = xyz(rad4);
    lastSamplePdf = thr4.w;
    flags = __float_as_uint(misc.z);
    seed = __float_as_uint(misc.w);
    scatterBounces = __float_as_uint(rad4.w);
    sampleIdx = med.w >> 16;
    depth = flags & PF_DEPTH_MASK;
    slot = __float_as_uint(hr.w);
    hitT = hr.x;

    // ---- infinite ground plane (checkInfinitePlaneIntersection, pathtrace_functions.h.slang:556-585): y = infinitePlaneDistance,
    //      hit from above only, when it lies in front of the geometry hit ----
    onPlane = false;
    catcher = false;
    if(F.fi.flags & B200PT_SCENE_USE_INFINITE_PLANE)
    {
      const float3 normal = f3(0, 1, 0);
      const float  planeHeight = F.fi.infinitePlaneDistance;
      const float  tGeom = (slot == 0xFFFFFFFFu) ? kInfinite : hitT;
      if(!(org.y <= planeHeight))
      {
        const float Dn = dot(dir, normal);
        if(!(fabsf(Dn) <= 1e-6f))
        {
          const float On = dot(org, normal);
          const float intersectionDist = (-On + planeHeight) / Dn;
          if(!(intersectionDist <= 0.0f || intersectionDist >= tGeom))
          {
            onPlane = true;
            hitT = intersectionDist;
            hit.pos = org + dir * hitT;
            hit.shadowPos = hit.pos;
            hit.nrm = normal;
            hit.geonrm = normal;
            hit.tangent = f3(1, 0, 0);
            hit.bitangent = f3(0, 0, 1);
            hit.color = f4(1, 1, 1, 1);
            hit.uv0 = hit.uv1 = f2(0.0f, 0.0f);
            hit.texelDensity = 0.0f;
            statAdd(&stats->shadedHits, 1ull);
            return true;
          }
        }
      }
    }

    if(slot == 0xFFFFFFFFu)
    {
      // ---- environment (gltf_pathtrace.slang:129-156) ----
      if(depth == 0)
      {
        flags &= ~PF_SOLID;  // tryPrimaryMissBackplate: pt.solid = false
        if(isFirstFrame(F, i))
          P.firstHit[i] = f4(dir, 0.0f);  // pt.firstHitPos = ray.Direction (pathtrace_functions.h.slang:950)
        if(F.fi.flags & B200PT_SCENE_USE_SOLID_BACKGROUND)
        {
          finalizeSample(P, F, i, f3(F.fi.backgroundColor[0], F.fi.backgroundColor[1], F.fi.backgroundColor[2]), false, seed, sampleIdx, qNext, cntNext, stats);
          return false;
        }
      }
      const float3 edir = rotateAxis(dir, f3(0, 1, 0), -F.fi.envRotation);
      const float4 env = sampleEnvTex(S, getSphericalUv(edir));
      float        misWeight = 1.0f;
      if(lastSamplePdf != kDirac)
      {
        float lw, ew;
        techniqueProbabilities(S, F, lw, ew);
        misWeight = lastSamplePdf / (lastSamplePdf + ew * env.w);
      }
      radiance += throughput * misWeight * (xyz(env) * F.fi.envIntensity);
      finalizeSample(P, F, i, radiance, (flags & PF_SOLID) != 0, seed, sampleIdx, qNext, cntNext, stats);
      return false;
    }

    // ---- hit-attribute fetch ----
    meta = S.triMeta[slot];
    nodeP = &S.nodes[meta.x & 0x0fffffffu];
    const b200pt_render_node& node = *nodeP;
    const ShadeRec            srec = loadShadeRec(S.shadeRecs + __ldg(&S.shadeIdx[slot]));
#ifdef B200PT_DEBUG
    // reference analogue: doDebug at pushConst.mouseCoord (gltf_pathtrace.slang:553-557)
    dbgPixel = ((float)(pixelOf(F, i) % (uint32_t)F.width) == F.pc.mouseCoord[0] && (float)pixelRow(F, pixelOf(F, i)) == F.pc.mouseCoord[1]);
    if(dbgPixel)
      printf("DBG hit t=%.9g rnode=%d prim=%d bary=%.9g %.9g org=%.9g %.9g %.9g dir=%.9g %.9g %.9g seed=%u depth=%d\n", hitT, (int)(meta.x & 0x0fffffffu), (int)meta.y, hr.y, hr.z,
             org.x, org.y, org.z, dir.x, dir.y, dir.z, seed, (int)depth);
#endif
    const float3              bary = f3(1.0f - hr.y - hr.z, hr.y, hr.z);
    hit = getHitState(srec, bary, node.worldToObject, node.objectToWorld, dir);
    statAdd(&stats->shadedHits, 1ull);
    return true;
  };
  // ---- section 2: material evaluation (three trilinear texture lookups), emission, unlit ----
  auto shadeMaterial = [&]() -> bool {
    worldFoot = (coneWidth + F.pc.pixelAngle * hitT) / fmaxf(fabsf(dot(hit.geonrm, -dir)), 1e-3f);
    int unlit = 0;
    if(onPlane)
    {
      // gltf_pathtrace.slang:169-173: defaultPbrMaterial(infinitePlaneBaseColor, metallic, roughness, N, N) (nvshaders, external:
      // restated -- GGX alpha = roughness^2 like evaluateMaterial, tangent frame from the normal; same in the oracle)
      pbrMat = defaultPbrMaterial();
      pbrMat.baseColor = f3(F.fi.infinitePlaneBaseColor[0], F.fi.infinitePlaneBaseColor[1], F.fi.infinitePlaneBaseColor[2]);
      pbrMat.metallic = F.fi.infinitePlaneMetallic;
      const float r = F.fi.infinitePlaneRoughness;
      pbrMat.roughness = f2(r * r, r * r);
      pbrMat.N = hit.nrm;
      pbrMat.Ng = hit.nrm;
      pbrMat.Nc = hit.nrm;
      pbrMat.T = xyz(makeFastTangent(hit.nrm));
      pbrMat.B = cross(pbrMat.N, pbrMat.T);
      if(F.fi.flags & B200PT_SCENE_INFINITE_PLANE_SHADOW_CATCHER)
      {
        // gltf_pathtrace.slang:175-186: the catcher returns before the first-hit captures, the roughness clamp and emission; its light
        // sample is drawn in the next section (the one sampleLights of this kernel), its second half runs after the shadow trace
        catcher = true;
        return true;
      }
    }
    else
    {
      const b200pt_render_node&    node = *nodeP;
      const int                    materialIndex = max(0, node.materialID);
      const float                  texGrad = worldFoot * hit.texelDensity * F.pc.texGradScale;
      const b200pt_shade_material& gmat = S.mats[materialIndex];
      pbrMat = evaluateMaterial<FEAT>(S, gmat, hit, (flags & PF_INSIDE) != 0, texGrad);
      unlit = gmat.unlit;
    }

    // firefly control: never get sharper than the roughest bounce so far (:267-268)
    misc.x = fmaxf(pbrMat.roughness.x, misc.x);
    misc.y = fmaxf(pbrMat.roughness.y, misc.y);
    pbrMat.roughness = f2(misc.x, misc.y);

    // first-hit capture for the NDC depth output of frame 0 (gltf_pathtrace.slang:228-232)
    if(depth == 0 && isFirstFrame(F, i))
      P.firstHit[i] = f4(hit.pos, 1.0f);
    // denoiser guides of the first hit (gltf_pathtrace.slang:240-263, the USE_GUIDE_SHADER part without the DLSS-only specular guides):
    // base colour and shading normal / roughness, stored as float16_t by the reference.  (maxRoughness is still 0 at depth 0, so the
    // clamp above left pbrMat.roughness as evaluateMaterial returned it.)
    if(depth == 0 && P.guideA && (F.pc.flags & B200PT_PT_USE_OPTIX_DENOISER))
    {
      auto h16 = [](float x) { return __half2float(__float2half_rn(x)); };
      P.guideA[i] = f4(h16(pbrMat.baseColor.x), h16(pbrMat.baseColor.y), h16(pbrMat.baseColor.z), h16(pbrMat.roughness.x));
      P.guideN[i] = f4(h16(pbrMat.N.x), h16(pbrMat.N.y), h16(pbrMat.N.z), 1.0f);
    }

    radiance += pbrMat.emissive * throughput;

    if(unlit > 0)
    {
      radiance += pbrMat.baseColor;
      finalizeSample(P, F, i, radiance, (flags & PF_SOLID) != 0, seed, sampleIdx, qNext, cntNext, stats);
      return false;
    }

    return true;
  };
  // ---- section 3: in-volume segment, light / environment sample ----
  auto shadeLight = [&]() -> bool {
    flags &= ~(PF_POST_VOLUME | PF_SHADOW_VALID | PF_SHADOW_INSIDE);

    // ---- in-volume segment (pathtrace_functions.h.slang:904-939, 605-672) ----
    if((FEAT & FEAT_VOLUME) && (flags & PF_INSIDE) && !catcher)
    {
      const VolumeMedium vm = unpackMedium(med);
      if(hasVolumeMedium(vm))
      {
        const float3 ext = vm.extinction, sc = vm.scatterCoefficient;
        bool         scattered = false;
        if(maxc(sc) > 0.001f)
        {
          const float maxExt = maxc(ext);
          const float scatterDist = -logf(fmaxf(rnd(seed), 1.0e-10f)) / maxExt;
          if(scatterDist < hitT)
          {
            throughput *= f3(1.0f) - (ext - sc) / maxExt;
            const float3 wi = dir;
            const float3 originBefore = org;
            org = org + dir * scatterDist;
            const float a = rnd(seed), b = rnd(seed);
            dir = sampleHenyeyGreenstein(f2(a, b), vm.scatterAnisotropy, wi);
            lastSamplePdf = henyeyGreensteinPdf(dot(wi, dir), vm.scatterAnisotropy);
            scattered = true;
            scatterBounces++;
            coneWidth += F.pc.pixelAngle * length(org - originBefore);
            // NEE at the scatter point (volumeScatterNEE)
            const DirectLight dl = sampleLights<FEAT>(S, F, org, seed);
            if(dl.pdf > 0.0f)
            {
              const float phasePdf = henyeyGreensteinPdf(dot(wi, dl.direction), vm.scatterAnisotropy);
              const float misWeight = dl.pdf / (dl.pdf + phasePdf);
              // reference: throughput * radianceOverPdf * misWeight * phasePdf * shadowFactor
              P.shC[i] = f4(throughput * dl.radianceOverPdf * misWeight * phasePdf, 0.0f);
              P.shO[i] = f4(org, dl.distance);
              P.shD[i] = f4(dl.direction, 0.0f);
              flags |= PF_SHADOW_VALID | PF_SHADOW_INSIDE;
            }
            flags |= PF_POST_VOLUME;
#ifdef B200PT_DEBUG
            if(dbgPixel)
              printf("DBG scatter n=%d o=%.9g %.9g %.9g d=%.9g %.9g %.9g thr=%.9g %.9g %.9g pdf=%.9g neeC=%.9g %.9g %.9g valid=%d seed=%u\n", (int)scatterBounces, org.x, org.y, org.z, dir.x, dir.y,
                     dir.z, throughput.x, throughput.y, throughput.z, lastSamplePdf, (flags & PF_SHADOW_VALID) ? P.shC[i].x : 0.f, (flags & PF_SHADOW_VALID) ? P.shC[i].y : 0.f,
                     (flags & PF_SHADOW_VALID) ? P.shC[i].z : 0.f, (int)((flags & PF_SHADOW_VALID) != 0), seed);
#endif
          }
          else
            throughput *= expv((f3(maxExt) - ext) * hitT);
        }
        else
          throughput *= expv(ext * -hitT);
        if(scattered)
        {
          P.rayO[i] = f4(org, coneWidth);
          P.rayD[i] = f4(normalize(dir), kInfinite);
          P.thr[i] = f4(throughput, lastSamplePdf);
          P.rad[i] = f4(radiance, __uint_as_float(scatterBounces));
          P.misc[i] = f4(misc.x, misc.y, __uint_as_float(flags), __uint_as_float(seed));
          queuePush(qPost, cntPost, i);
          if(flags & PF_SHADOW_VALID)
            queuePush(qShadow, cntShadow, i);
          return false;
        }
      }
    }

    coneWidth = worldFoot;

    // ---- next-event estimation: one light-or-environment sample, MIS (:316-351) ----
    directLight = sampleLights<FEAT>(S, F, hit.pos, seed);
    if(catcher)
    {
      // handleShadowCatcher, first half (:511-523): the light sample and its shadow ray -- from the plane point itself, unbounded.
      // The shadow factor comes back through the shadow / any-hit kernels in shC; finishPost continues with the second half.
      flags |= PF_CATCHER;
      if(dot(directLight.direction, hit.nrm) > 0.0f && directLight.pdf != 0.0f)
      {
        P.shO[i] = f4(hit.pos, kInfinite);
        P.shD[i] = f4(directLight.direction, 0.0f);
        P.shC[i] = f4(1.0f, 1.0f, 1.0f, 0.0f);
        flags |= PF_SHADOW_VALID;
      }
      P.rayO[i] = f4(hit.pos, coneWidth);  // the incoming direction stays in rayD: the second half looks the environment up along it
      P.misc[i] = f4(misc.x, misc.y, __uint_as_float(flags), __uint_as_float(seed));
      queuePush(qPost, cntPost, i);
      if(flags & PF_SHADOW_VALID)
        queuePush(qShadow, cntShadow, i);
      return false;
    }
    nextEventValid = (dot(directLight.direction, hit.nrm) > 0.0f || pbrMat.diffuseTransmissionFactor > 0.0f) && directLight.pdf != 0.0f;
    return true;
  };
  // ---- section 4: BSDF evaluation for the light sample, BSDF sampling, next ray + shadow ray ----
  auto shadeBsdf = [&]() {
    float3 contribution = f3(0.0f);
#ifdef B200PT_DEBUG
    if(dbgPixel)
      printf("DBG shade pos=%.9g %.9g %.9g nrm=%.9g %.9g %.9g gn=%.9g %.9g %.9g N=%.9g %.9g %.9g rough=%.9g %.9g metal=%.9g base=%.9g %.9g %.9g L=%.9g %.9g %.9g lpdf=%.9g valid=%d seed=%u\n",
             hit.pos.x, hit.pos.y, hit.pos.z, hit.nrm.x, hit.nrm.y, hit.nrm.z, hit.geonrm.x, hit.geonrm.y, hit.geonrm.z, pbrMat.N.x, pbrMat.N.y, pbrMat.N.z, pbrMat.roughness.x,
             pbrMat.roughness.y, pbrMat.metallic, pbrMat.baseColor.x, pbrMat.baseColor.y, pbrMat.baseColor.z, directLight.direction.x, directLight.direction.y,
             directLight.direction.z, directLight.pdf, (int)nextEventValid, seed);
#endif
    if(nextEventValid)
    {
      const float    a = rnd(seed), b = rnd(seed), c = rnd(seed);
      const BsdfEval ev = bsdfEvaluate<FEAT>(pbrMat, -dir, directLight.direction, f3(a, b, c));
      if(ev.pdf > 0.0f)
      {
        const float  misWeight = (directLight.pdf == kDirac) ? 1.0f : directLight.pdf / (directLight.pdf + ev.pdf);
        const float3 w = throughput * directLight.radianceOverPdf * misWeight;
        contribution += w * ev.bsdf_diffuse;
        contribution += w * ev.bsdf_glossy;
      }
    }

    // ---- BSDF sampling: next direction + throughput (:357-416) ----
    {
      const float      a = rnd(seed), b = rnd(seed), c = rnd(seed);
      const BsdfSample sd = bsdfSample<FEAT>(pbrMat, -dir, f3(a, b, c));
#ifdef B200PT_DEBUG
      if(dbgPixel)
        printf("DBG sample xi=%.9g %.9g %.9g k2=%.9g %.9g %.9g bop=%.9g %.9g %.9g pdf=%.9g ev=%d contrib=%.9g %.9g %.9g\n", a, b, c, sd.k2.x, sd.k2.y, sd.k2.z, sd.bsdf_over_pdf.x,
               sd.bsdf_over_pdf.y, sd.bsdf_over_pdf.z, sd.pdf, sd.event_type, contribution.x, contribution.y, contribution.z);
#endif
      throughput *= sd.bsdf_over_pdf;
      dir = sd.k2;
      lastSamplePdf = sd.pdf;
      if(sd.event_type != BSDF_EVENT_ABSORB)
      {
        const float3 offsetDir = dot(dir, hit.geonrm) > 0 ? hit.geonrm : -hit.geonrm;
        org = safeOffsetRay(hit.pos, offsetDir);
        if((FEAT & (FEAT_TRANSMISSION | FEAT_DIFFUSE_TRANSMISSION)) && (sd.event_type & BSDF_EVENT_TRANSMISSION))
        {
          flags ^= PF_INSIDE;
          if((FEAT & FEAT_VOLUME) && (flags & PF_INSIDE))
            med = packMedium(makeVolumeMedium(pbrMat), med.w >> 16);
        }
      }
      else
        depth = (uint32_t)F.pc.maxDepth;
    }

    // ---- shadow ray for the delayed NEE visibility test (:418-426) ----
    if(nextEventValid)
    {
      const bool   forward = dot(directLight.direction, hit.nrm) > 0.0f;
      const float3 sDir = forward ? hit.geonrm : -hit.geonrm;
      const float3 sBase = forward ? hit.shadowPos : hit.pos;
      P.shO[i] = f4(safeOffsetRay(sBase, sDir), directLight.distance);
      P.shD[i] = f4(directLight.direction, 0.0f);
      P.shC[i] = f4(contribution, 0.0f);
      flags |= PF_SHADOW_VALID;
    }

    flags = (flags & ~PF_DEPTH_MASK) | (depth & PF_DEPTH_MASK);
    P.rayO[i] = f4(org, coneWidth);
    P.rayD[i] = f4(normalize(dir), kInfinite);
    P.thr[i] = f4(throughput, lastSamplePdf);
    P.rad[i] = f4(radiance, __uint_as_float(scatterBounces));
    P.misc[i] = f4(misc.x, misc.y, __uint_as_float(flags), __uint_as_float(seed));
    P.medium[i] = med;
    queuePush(qPost, cntPost, i);
    if(flags & PF_SHADOW_VALID)
      queuePush(qShadow, cntShadow, i);
  };
  for(uint32_t base = blockIdx.x * blockDim.x; base < count; base += stride)
  {
    bool alive = base + threadIdx.x < count;
    __syncthreads();
    if(alive)
      alive = shadeLoad(base + threadIdx.x);
    if(alive)
      alive = shadeMaterial();
    if(alive)
      alive = shadeLight();
    if(alive)
      shadeBsdf();
  }
}

// pathTrace() tail for every path that survived shading: delayed NEE visibility (TraceShadow), Russian
// roulette, depth++ (gltf_pathtrace.slang:462-485).  Same persistent-warp scheme as k_trace; paths without a
// shadow ray finish immediately and their lanes are refilled.
__device__ void finishPost(const PathState& P, const DevScene& S, const FrameParams& F, uint32_t i, uint32_t flags, uint32_t seed, bool haveShadow, float3 Tfac,
                           uint32_t* qNext, uint32_t* cntNext, DevStats* stats)
{
  const float4 misc = P.misc[i];
  const float4 rad4 = P.rad[i];
  float3       radiance = xyz(rad4);
  const float4 thr4 = P.thr[i];
  float3       throughput = xyz(thr4);
  if(flags & PF_CATCHER)
  {
    // handleShadowCatcher, second half (pathtrace_functions.h.slang:525-553): lit plane points show the environment behind them and
    // end the path; shadowed ones show it darkened and continue with bsdfSampleSimple -- eEarlyContinue: no roulette, no depth++
    const float3 shadowFactor = haveShadow ? xyz(P.shC[i]) * Tfac : f3(1.0f);
    const float4 ro = P.rayO[i];
    const float3 hitPos = xyz(ro), dir = xyz(P.rayD[i]);
    const float4 env = sampleEnvTex(S, getSphericalUv(rotateAxis(dir, f3(0, 1, 0), -F.fi.envRotation)));
    const float3 envColor = xyz(env) * F.fi.envIntensity;
    flags &= ~(PF_CATCHER | PF_POST_VOLUME | PF_SHADOW_VALID | PF_SHADOW_INSIDE);
    if(shadowFactor.x == 1.0f && shadowFactor.y == 1.0f && shadowFactor.z == 1.0f)
    {
      float misWeight = 1.0f;
      if(thr4.w != kDirac)
      {
        float lw, ew;
        techniqueProbabilities(S, F, lw, ew);
        misWeight = thr4.w / (thr4.w + ew * env.w);
      }
      radiance += throughput * misWeight * envColor;
      finalizeSample(P, F, i, radiance, (flags & PF_SOLID) != 0, seed, P.medium[i].w >> 16, qNext, cntNext, stats);
      return;
    }
    radiance += envColor * shadowFactor;
    radiance -= envColor * (f3(1.0f) - shadowFactor) * F.fi.shadowCatcherDarkenAmount;
    PbrMaterial  pm = defaultPbrMaterial();  // the plane's material, as k_shade built it (gltf_pathtrace.slang:169-173)
    const float3 n = f3(0, 1, 0);
    pm.baseColor = f3(F.fi.infinitePlaneBaseColor[0], F.fi.infinitePlaneBaseColor[1], F.fi.infinitePlaneBaseColor[2]);
    pm.metallic = F.fi.infinitePlaneMetallic;
    const float r = F.fi.infinitePlaneRoughness;
    pm.roughness = f2(r * r, r * r);
    pm.N = pm.Ng = pm.Nc = n;
    pm.T = xyz(makeFastTangent(n));
    pm.B = cross(pm.N, pm.T);
    const float      a = rnd(seed), b = rnd(seed), c = rnd(seed);
    const BsdfSample sd = bsdfSampleSimple(pm, -dir, f3(a, b, c));
    if(sd.event_type == BSDF_EVENT_ABSORB)
    {
      finalizeSample(P, F, i, radiance, (flags & PF_SOLID) != 0, seed, P.medium[i].w >> 16, qNext, cntNext, stats);
      return;
    }
    const float3 offsetDir = dot(sd.k2, n) > 0 ? n : -n;
    throughput *= sd.bsdf_over_pdf;
    P.rayO[i] = f4(safeOffsetRay(hitPos, offsetDir), ro.w);
    P.rayD[i] = f4(normalize(sd.k2), kInfinite);
    P.thr[i] = f4(throughput, sd.pdf);
    P.rad[i] = f4(radiance, rad4.w);
    P.misc[i] = f4(misc.x, misc.y, __uint_as_float(flags), __uint_as_float(seed));
    queuePush(qNext, cntNext, i);
    return;
  }
  if(haveShadow)
    radiance += xyz(P.shC[i]) * Tfac;
  uint32_t     depth = flags & PF_DEPTH_MASK;
  bool         alive = true, thrDirty = false;
  if(flags & PF_POST_VOLUME)
  {
    // in-volume Russian roulette only after VOLUME_FREE_BUDGET scatters (pathtrace_functions.h.slang:925-931)
    if(__float_as_uint(rad4.w) >= 64u)
    {
      const float rrPcont = fminf(maxc(throughput) + 0.001f, 0.95f);
      if(rnd(seed) >= rrPcont)
        alive = false;
      else
      {
        throughput /= rrPcont;
        thrDirty = true;
      }
    }
  }
  else
  {
    // surface Russian roulette from depth 3 (gltf_pathtrace.slang:476-485)
    if(depth >= 3u)
    {
      const float rrPcont = fminf(maxc(throughput) + 0.001f, 0.95f);
      if(rnd(seed) >= rrPcont)
        alive = false;
      else
      {
        throughput /= rrPcont;
        thrDirty = true;
      }
    }
    if(alive)
    {
      depth++;
      if((int)depth >= F.pc.maxDepth)
        alive = false;
    }
  }
  if(!alive)
  {
    finalizeSample(P, F, i, radiance, (flags & PF_SOLID) != 0, seed, P.medium[i].w >> 16, qNext, cntNext, stats);
    return;
  }
  flags = (flags & ~(PF_DEPTH_MASK | PF_POST_VOLUME | PF_SHADOW_VALID | PF_SHADOW_INSIDE)) | (depth & PF_DEPTH_MASK);
  if(haveShadow)
    P.rad[i] = f4(radiance, rad4.w);
  if(thrDirty)
    P.thr[i] = f4(throughput, thr4.w);
  P.misc[i] = f4(misc.x, misc.y, __uint_as_float(flags), __uint_as_float(seed));
  queuePush(qNext, cntNext, i);
}

// IRaytracer::TraceShadow, geometry part, for every path with a pending NEE shadow ray: ONE walk of the scene tree along
// the whole segment; any FORCE_OPAQUE occluder ends the query (raytracer_interface.h.slang:181-184), otherwise the kCand
// nearest non-opaque candidates are written out for k_alpha<true>.  Same persistent-warp scheme as k_trace.
template <bool OMM>
__global__ void __launch_bounds__(128, kTraceMinBlocks) k_shadow(PathState P, DevScene S, const uint32_t* __restrict__ q, const uint32_t* __restrict__ cntIn,
                                                                        uint32_t* workCounter, uint32_t* qAlpha, uint32_t* cntAlpha, DevStats* stats,
                                                                        int refillThreshold, int postponeShift, int mode)
{
  __shared__ Cand s_cand[kCand * 128];
  Cand* const     cand = &s_cand[threadIdx.x];
  constexpr int   cs = 128;
  const bool      cont = (mode & TRACE_CONT) != 0;
  const uint32_t  count = *cntIn;
  TravState       T;
  uint2           stack[TravState::kStackSize];
  int             path = -1;  // -1: lane needs work, -2: queue exhausted
  int             phase = 0;  // 0: occlusion query against the opaque-only tree, 1: candidates from the non-opaque tree
  bool            travDone = false;
  for(;;)
  {
    __syncwarp();
    if(path >= 0 && travDone)
    {
      travDone = false;
      T.flushCounters(&stats->nodesVisited, &stats->trisTested);
      if(T.overflow)
        atomicOr(&stats->errorFlags, 1ull);
      if(phase == 0 && T.best.slot == 0xFFFFFFFFu && S.hasAlpha)
      {
        // no opaque occluder: the non-opaque candidates of the segment, nearest first
        // With opacity micromaps an OPAQUE micro-triangle anywhere on the segment ends the query like a FORCE_OPAQUE occluder
        // (a committed hit, raytracer_interface.h.slang:181-184), so the walk must not stop looking behind the 4th candidate.
        phase = 1;
        T.init(S.bvhA, T.org, T.dir, 0.0f, T.tmax, false, true, false, 0.f, 0u, !OMM);
      }
      else
      {
        uint2 info = make_uint2(0u, 0u);
        if(T.best.slot != 0xFFFFFFFFu)
          info.x = 0x80000000u;  // an opaque occluder ended the query (raytracer_interface.h.slang:181-184)
        else
        {
          const int n = T.collectN;
#pragma unroll
          for(int i = 0; i < kCand; i++)
            if(i < n)
            {
              const Cand c = cand[i * cs];
              P.cand[i][path] = f4(c.t, c.u, c.v, __uint_as_float(c.slot));
            }
          info = make_uint2((uint32_t)n, n > 0 ? cand[(n - 1) * cs].gid : 0u);
        }
        P.candInfo[path] = info;
        // (a continuation path always goes back to k_alpha: its running transmission is parked and must be folded)
        if((info.x != 0u && info.x != 0x80000000u) || cont)
          queuePush(qAlpha, cntAlpha, (uint32_t)path);
        path = -1;
      }
    }
    __syncwarp();
    {
      const bool     need = (path == -1);
      const uint32_t k = fetchWork(need, workCounter, count);
      if(need)
      {
        if(k == 0xFFFFFFFFu)
          path = -2;
        else
        {
          path = (int)q[k];
          const float4 so = P.shO[path];
          const float4 sd = P.shD[path];
          if(!cont)
          {
            phase = 0;
            T.init(S.bvhO, xyz(so), xyz(sd), 0.0f, so.w, false, true, false, 0.f, 0u, false);
          }
          else
          {
            phase = 1;
            T.init(S.bvhA, xyz(so), xyz(sd), 0.0f, so.w, false, true, true, P.cand[kCand - 1][path].x, P.candInfo[path].y, true);
          }
        }
      }
    }
    if(__all_sync(0xffffffffu, path == -2))
      break;
    for(;;)
    {
#ifdef B200PT_COUNT_TRAVERSAL
      {
        const unsigned busy = __ballot_sync(0xffffffffu, path >= 0 && !travDone);
        if((threadIdx.x & 31) == 0)
        {
          atomicAdd(&stats->warpIters, 1ull);
          atomicAdd(&stats->busyLaneIters, (unsigned long long)__popc(busy));
        }
      }
#endif
      if(path >= 0 && !travDone)
        travDone = T.step<kCand, false, OMM, 2>(stack, postponeShift, cand, cs, S.bvhA.ommRef, S.bvhA.ommData);  // (only non-opaque triangles consult it: phase 1)
      if(__popc(__ballot_sync(0xffffffffu, path >= 0 && !travDone)) < refillThreshold)
        break;
    }
  }
  if(blockIdx.x == 0 && threadIdx.x == 0 && !cont)
    atomicAdd(&stats->shadowRays, (unsigned long long)count);
}

// the walk kernels have an instantiation for scenes with opacity micromaps (omm.cuh) and one without the lookup
#define WALK_KERNEL(K, grid, ...)                  \
  do                                               \
  {                                                \
    if(omm)                                        \
      K<true><<<grid, 128, 0, st>>>(__VA_ARGS__);  \
    else                                           \
      K<false><<<grid, 128, 0, st>>>(__VA_ARGS__); \
  } while(0)

// pathTrace() tail for every path that survived shading (gltf_pathtrace.slang:462-485), one thread per path: the
// delayed NEE contribution (already scaled by the any-hit transmission in k_alpha<true>; an opaque occluder
// zeroes it here), Russian roulette and depth++ in finishPost.
__global__ void __launch_bounds__(256) k_resolve(PathState P, DevScene S, const __grid_constant__ FrameParams F, const uint32_t* __restrict__ q, const uint32_t* __restrict__ cntIn,
                                                 uint32_t* qNext, uint32_t* cntNext, DevStats* stats)
{
  const uint32_t count = *cntIn;
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
  {
    const uint32_t path = q[k];
    const float4   misc = P.misc[path];
    const uint32_t flags = __float_as_uint(misc.z);
    const uint32_t seed = __float_as_uint(misc.w);
    const bool     haveShadow = (flags & PF_SHADOW_VALID) != 0;
    float3         vis = f3(1.0f);
    if(haveShadow && (P.candInfo[path].x & 0x80000000u))
      vis = f3(0.0f);
#ifdef B200PT_DEBUG
    if(haveShadow && (float)(pixelOf(F, path) % (uint32_t)F.width) == F.pc.mouseCoord[0] && (float)pixelRow(F, pixelOf(F, path)) == F.pc.mouseCoord[1])
      printf("DBG shadow occluded=%d\n", (int)(vis.x == 0.0f));
#endif
    finishPost(P, S, F, path, flags, seed, haveShadow, vis, qNext, cntNext, stats);
  }
}

// processPixel tail: mean over the frame's samples + running mean over frames (gltf_pathtrace.slang:596,619-630); on the
// first frame also the NDC depth of the last sample's first hit (:600-616; Vulkan [0,1] range, 1 = far / miss)
__global__ void __launch_bounds__(256) k_accumulate(PathState P, const __grid_constant__ FrameParams F, float4* __restrict__ accum, float* __restrict__ ndcDepth)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < F.pixels; i += stride)
  {
    float4 img = f4(0.f, 0.f, 0.f, 0.f);
    // the frames of a batch are folded in frame order, each with the sample counts its own push constants would have carried
    for(int b = 0; b < F.batch; b++)
    {
      const float4 c = P.pixSum[i + (uint32_t)b * F.pixels] / (float)F.pc.numSamples;
      if(b == 0 && (F.pc.flags & B200PT_PT_FIRST_FRAME))
      {
        img = c;
        if(ndcDepth)
        {
          const float4 fh = P.firstHit[i];
          float        d = 1.0f;
          if(fh.w > 0.0f)
          {
            const Mat4&  vp = *reinterpret_cast<const Mat4*>(F.fi.viewProjMatrix);
            const float4 clip = mul_vM(f4(fh.x, fh.y, fh.z, 1.0f), vp);
            d = clip.z / clip.w;
          }
          ndcDepth[i] = d;
        }
      }
      else
      {
        if(b == 0)
          img = accum[i];
        const int    totalSamples = F.pc.totalSamples + b * F.pc.numSamples;
        const float  total = (float)totalSamples, n = (float)F.pc.numSamples;
        const float  after = (float)(totalSamples + F.pc.numSamples);
        const float4 old = img;
        img = f4((old.x * total + c.x * n) / after, (old.y * total + c.y * n) / after, (old.z * total + c.z * n) / after, (old.w * total + c.w * n) / after);
      }
    }
    accum[i] = img;
  }
}

// OutputImage::eOptixAlbedoNormal (gltf_pathtrace.slang:653-670): per pixel the LAST sample's guide albedo and its shading normal in
// camera space, compressed to 32 bits.  compressUnitVec is nvshaders code (external): restated as the octahedral 2 x 16-bit encoding it
// implements (Engelhardt & Dachsbacher 2008): project onto |x| + |y| + |z| = 1, fold the lower hemisphere, 16 bits per axis.
PT_HD uint32_t compressUnitVec(float3 nv)
{
  if(!(fabsf(nv.x) < 3.0e38f))  // NaN / infinity
    return ~0u;
  const float d = 32767.0f / (fabsf(nv.x) + fabsf(nv.y) + fabsf(nv.z));
  int         x = (int)roundf(nv.x * d), y = (int)roundf(nv.y * d);
  if(nv.z < 0.0f)
  {
    const int maskx = x >> 31, masky = y >> 31;
    const int tmp = 32767 + maskx + masky, tmpx = x;
    x = (tmp - (y ^ masky)) ^ maskx;
    y = (tmp - (tmpx ^ maskx)) ^ masky;
  }
  const uint32_t packed = ((uint32_t)(y + 32767) << 16) | (uint32_t)(x + 32767);
  return packed == ~0u ? ~1u : packed;
}

__global__ void __launch_bounds__(256) k_guide(PathState P, const __grid_constant__ FrameParams F, float4* __restrict__ guide)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < F.pixels; i += stride)
  {
    const uint32_t slot = i + (uint32_t)(F.batch - 1) * F.pixels;  // the newest frame of the batch
    const float4   a = P.guideA[slot], n = P.guideN[slot];
    float3         camN = f3(0.0f, 0.0f, 1.0f);  // primary miss: a valid forward-facing normal (:658-660)
    if(n.w > 0.0f)
    {
      // mul(float3x3(viewMatrix), worldNormal) on the glm bytes (SURVEY.md section 8, convention note): M_glm^T * n
      const float* m = F.fi.viewMatrix;
      camN = normalize(f3((m[0] * n.x + m[1] * n.y) + m[2] * n.z, (m[4] * n.x + m[5] * n.y) + m[6] * n.z, (m[8] * n.x + m[9] * n.y) + m[10] * n.z));
    }
    guide[i] = f4(a.x, a.y, a.z, __uint_as_float(compressUnitVec(camN)));
  }
}

// traceSelectionRay (pathtrace_functions.h.slang:813-820) for every pixel of the first frame: the pixel-centre ray
// (no jitter, no depth of field), IRaytracer::TraceLow semantics (raytracer_interface.h.slang:124-137: every triangle
// opaque, no culling), object id = render node + 1, 0 on a miss.  One walk per thread; runs once per accumulation.
__global__ void __launch_bounds__(128) k_select(DevScene S, const __grid_constant__ FrameParams F, uint32_t* __restrict__ objectId, DevStats* stats)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  const Mat4&    projI = *reinterpret_cast<const Mat4*>(F.fi.projInv);
  const Mat4&    viewI = *reinterpret_cast<const Mat4*>(F.fi.viewInv);
  const bool     ortho = (F.fi.flags & B200PT_SCENE_IS_ORTHOGRAPHIC) != 0;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < F.pixels; i += stride)
  {
    const uint32_t x = i % (uint32_t)F.width;
    const uint32_t y = pixelRow(F, i);
    const float2   clip = f2(((float)x + 0.5f) / F.fi.imageSize[0] * 2.0f - 1.0f, ((float)y + 0.5f) / F.fi.imageSize[1] * 2.0f - 1.0f);
    float4         vc = mul_vM(f4(clip.x, clip.y, -1.0f, 1.0f), projI);
    vc = vc / vc.w;
    float3 org, dir;
    if(ortho)
    {
      org = xyz(mul_vM(vc, viewI));
      dir = normalize(xyz(mul_vM(f4(0, 0, -1, 0), viewI)));
    }
    else
    {
      org = f3(viewI.m[12], viewI.m[13], viewI.m[14]);
      dir = normalize(xyz(mul_vM(vc, viewI)) - org);
    }
    TravState T;
    uint2     stack[TravState::kStackSize];
    Cand      cand[1];
    T.init(S.bvh, org, dir, 0.0f, kInfinite, false, false, false, 0.f, 0u);
    while(!T.step<1, true>(stack, 2, cand, 1))
    {
    }
    if(T.overflow)
      atomicOr(&stats->errorFlags, 1ull);
    objectId[i] = (T.best.slot != 0xFFFFFFFFu) ? (S.triMeta[T.best.slot].x & 0x0fffffffu) + 1u : 0u;
  }
}

// ---- BVH construction on the device (lbvh.cuh) --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lbvh_bounds(LbvhWork W)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i < W.m)
    lbvhBounds(i, W);
}
__global__ void __launch_bounds__(256) k_lbvh_morton(LbvhWork W)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i < W.M)
    lbvhMorton(i, W);
}
__global__ void __launch_bounds__(256) k_lbvh_bitonic(unsigned long long* keys, uint32_t n, uint32_t j, uint32_t k)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if(t < n)
    bitonicStep(t, keys, j, k);
}
__global__ void __launch_bounds__(256) k_lbvh_hierarchy(LbvhWork W)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i + 1 < W.m)
    lbvhHierarchy(i, W);
}
__global__ void __launch_bounds__(256) k_lbvh_fit(LbvhWork W)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i < W.m)
    lbvhFit(i, W);
}
__global__ void __launch_bounds__(128) k_lbvh_emit(LbvhWork W, const int2* queueIn, uint32_t count, int2* queueOut)
{
  const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
  if(q < count)
    lbvhEmit(q, W, queueIn, queueOut);
}

// ---- BVH refit after a transform update (refit.cuh) ------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_refit_tris(float* tris, uint2* triMeta, uint32_t n, const b200pt_render_node* nodes, const DevPrim* prims)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    refitTriangle(i, tris, triMeta, nodes, prims);
}

__global__ void __launch_bounds__(128) k_refit_level(float* nodes, const float* tris, float4* nodeBox, uint32_t first, uint32_t count)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
    refitNode(first + i, nodes, tris, nodeBox);
}

// ---- tone mapping + 8-bit encode (tonemap.cuh): HBM-bound, 16 B read + 4 B written per pixel (+ 16 B read for the histogram) ----
__global__ void __launch_bounds__(256) k_tm_histogram(const float4* __restrict__ img, uint32_t n, uint32_t* __restrict__ hist)
{
  __shared__ uint32_t s_h[kTmBins];
  for(int i = threadIdx.x; i < kTmBins; i += blockDim.x)
    s_h[i] = 0u;
  __syncthreads();
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
  {
    const float4 c = __ldg(&img[i]);
    atomicAdd(&s_h[tmBin(0.2126f * c.x + 0.7152f * c.y + 0.0722f * c.z)], 1u);
  }
  __syncthreads();
  for(int i = threadIdx.x; i < kTmBins; i += blockDim.x)
    if(s_h[i])
      atomicAdd(&hist[i], s_h[i]);
}

// log-average luminance over the bins above black -> exposure factor (integer counts, fixed summation order: deterministic)
__global__ void k_tm_exposure(const uint32_t* __restrict__ hist, float baseExposure, float* __restrict__ out)
{
  if(blockIdx.x == 0 && threadIdx.x == 0)
  {
    double sum = 0.0, cnt = 0.0;
    for(int b = 1; b < kTmBins; b++)
    {
      const double centre = (double)kTmMinLog + ((double)b + 0.5) * (double)(kTmMaxLog - kTmMinLog) / (double)kTmBins;
      sum += centre * (double)hist[b];
      cnt += (double)hist[b];
    }
    *out = cnt > 0.0 ? baseExposure * (float)(0.18 / exp2(sum / cnt)) : baseExposure;
  }
}

__global__ void __launch_bounds__(256) k_tonemap(const float4* __restrict__ img, uchar4* __restrict__ out, int width, int rows, int y0, int fullHeight,
                                                 const __grid_constant__ b200pt_tonemapper tm, const float* __restrict__ exposure)
{
  const uint32_t n = (uint32_t)width * (uint32_t)rows, stride = gridDim.x * blockDim.x;
  const float    ex = *exposure;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
  {
    const float4 c = __ldg(&img[i]);
    const int    x = (int)(i % (uint32_t)width), y = y0 + (int)(i / (uint32_t)width);
    const float3 r = tonemapPixel(tm, ex, f3(c.x, c.y, c.z), ((float)x + 0.5f) / (float)width, ((float)y + 0.5f) / (float)fullHeight);
    out[i] = make_uchar4((unsigned char)tmUnorm8(r.x), (unsigned char)tmUnorm8(r.y), (unsigned char)tmUnorm8(r.z), (unsigned char)tmUnorm8(c.w));
  }
}

// ---- animation feed (animate.cuh): morph.comp.slang / skinning.comp.slang, one thread per vertex like the reference's
// ANIMATION_WORKGROUP_SIZE = 256 dispatches; HBM-bound (<= 72 B read + 40 B written per vertex, matrices stay in L1) -------------
__global__ void __launch_bounds__(256) k_morph(MorphTaskDev T)
{
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if(v < T.vertexCount)
    morphVertex(T, v);
}

__global__ void __launch_bounds__(256) k_skin(SkinTaskDev T)
{
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if(v < T.vertexCount)
    skinVertex(T, v);
}

__global__ void __launch_bounds__(256) k_propagate_level(const float* __restrict__ local, float* world, const int* __restrict__ parents, const int* __restrict__ topo,
                                                         uint32_t levelOffset, uint32_t levelCount)
{
  const uint32_t ti = blockIdx.x * blockDim.x + threadIdx.x;
  if(ti < levelCount)
    propagateNode(local, world, parents, topo, levelOffset, ti);
}

__global__ void __launch_bounds__(256) k_update_render_nodes(const float* __restrict__ world, const RenderNodeMapping* __restrict__ mappings,
                                                             const float* __restrict__ instLocal, b200pt_render_node* out, uint32_t n)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i < n)
    updateRenderNode(world, mappings, instLocal, out, i);
}

__global__ void __launch_bounds__(256) k_regather_shade(ShadeRec* recs, DevPrim P, uint32_t triCount)
{
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if(t < triCount)
    regatherShadeRec(recs + t, P, t);
}

// ---- ray-level API (parity tests / traversal micro-benchmark): the rays run through the PRODUCTION kernels
// (k_trace / k_shadow -> k_alpha -> continuation round -> k_alpha) on a scratch path pool -------------------------
__global__ void __launch_bounds__(256) k_rays_load(PathState P, const float4* __restrict__ rays, uint32_t n, const uint32_t* __restrict__ seeds, uint32_t* q, uint32_t* cnt,
                                                   int shadow)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
  {
    const float4 o = rays[i * 2], d = rays[i * 2 + 1];
    if(!shadow)
    {
      P.rayO[i] = o;  // .w = tmin (TRACE_TMIN)
      P.rayD[i] = d;  // .w = tmax
    }
    else
    {
      P.shO[i] = f4(o.x, o.y, o.z, d.w);
      P.shD[i] = f4(d.x, d.y, d.z, 0.0f);
      P.shC[i] = f4(1.0f, 1.0f, 1.0f, 0.0f);
    }
    P.misc[i] = f4(0.0f, 0.0f, __uint_as_float(shadow ? PF_SHADOW_VALID : 0u), __uint_as_float(seeds ? seeds[i] : 0u));
    P.candInfo[i] = make_uint2(0u, 0u);
    q[i] = i;
  }
  if(blockIdx.x == 0 && threadIdx.x == 0)
    *cnt = n;
}

__global__ void __launch_bounds__(256) k_rays_store(PathState P, DevScene S, uint32_t n, float* __restrict__ out, uint32_t* seeds, int shadow)
{
  const uint32_t stride = gridDim.x * blockDim.x;
  for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
  {
    if(seeds)
      seeds[i] = __float_as_uint(P.misc[i].w);
    if(shadow)
    {
      const float4 c = P.shC[i];
      const bool   occluded = (P.candInfo[i].x & 0x80000000u) != 0;
      out[i * 3] = occluded ? 0.0f : c.x;
      out[i * 3 + 1] = occluded ? 0.0f : c.y;
      out[i * 3 + 2] = occluded ? 0.0f : c.z;
      continue;
    }
    const float4   h = P.hit[i];
    const uint32_t slot = __float_as_uint(h.w);
    float*         o = out + (size_t)i * 6;
    int            rnode = -1, rprim = -1, primId = -1;
    float          t = kInfinite, u = 0.f, v = 0.f;
    if(slot != 0xFFFFFFFFu)
    {
      const uint2 meta = S.triMeta[slot];
      rnode = (int)(meta.x & 0x0fffffffu);
      rprim = S.nodes[rnode].renderPrimID;
      primId = (int)meta.y;
      t = h.x;
      u = h.y;
      v = h.z;
    }
    o[0] = t;
    o[1] = __int_as_float(rnode);
    o[2] = __int_as_float(rprim);
    o[3] = __int_as_float(primId);
    o[4] = u;
    o[5] = v;
  }
}

// packing of the BSDF test records: vk_gltf_renderer_b200/bsdf_io.py
__device__ PbrMaterial unpackTestMaterial(const float* p)
{
  PbrMaterial m;
  m.baseColor = f3(p[0], p[1], p[2]);
  m.opacity = 1.0f;
  m.roughness = f2(p[3], p[4]);
  m.metallic = p[5];
  m.emissive = f3(0.0f);
  m.N = f3(p[6], p[7], p[8]);
  m.T = f3(p[9], p[10], p[11]);
  m.B = f3(p[12], p[13], p[14]);
  m.Ng = f3(p[15], p[16], p[17]);
  m.ior1 = p[18];
  m.ior2 = p[19];
  m.specular = p[20];
  m.specularColor = f3(p[21], p[22], p[23]);
  m.transmission = p[24];
  m.attenuationColor = f3(1.0f);
  m.attenuationDistance = 1.0f;
  m.thickness = p[25];
  m.clearcoat = p[26];
  m.clearcoatRoughness = p[27];
  m.Nc = m.N;
  m.iridescence = p[28];
  m.iridescenceIor = p[29];
  m.iridescenceThickness = p[30];
  m.sheenColor = f3(p[31], p[32], p[33]);
  m.sheenRoughness = p[34];
  m.diffuseTransmissionFactor = p[35];
  m.diffuseTransmissionColor = f3(p[36], p[37], p[38]);
  m.scatterCoefficient = f3(0.0f);
  m.scatterAnisotropy = 0.0f;
  m.dispersion = 0.0f;
  m.retroreflection = 0.0f;
  return m;
}

__global__ void k_bsdf_eval(const float* __restrict__ in, uint32_t n, float* __restrict__ out)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n)
    return;
  const float*      p = in + (size_t)i * 48;
  const PbrMaterial m = unpackTestMaterial(p);
  const BsdfEval    d = bsdfEvaluate<FEAT_ALL>(m, f3(p[39], p[40], p[41]), f3(p[42], p[43], p[44]), f3(p[45], p[46], p[47]));
  float*            q = out + (size_t)i * 8;
  q[0] = d.bsdf_diffuse.x;
  q[1] = d.bsdf_diffuse.y;
  q[2] = d.bsdf_diffuse.z;
  q[3] = d.bsdf_glossy.x;
  q[4] = d.bsdf_glossy.y;
  q[5] = d.bsdf_glossy.z;
  q[6] = d.pdf;
  q[7] = 0.f;
}

__global__ void k_bsdf_sample(const float* __restrict__ in, uint32_t n, float* __restrict__ out)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i >= n)
    return;
  const float*      p = in + (size_t)i * 48;
  const PbrMaterial m = unpackTestMaterial(p);
  const BsdfSample  d = bsdfSample<FEAT_ALL>(m, f3(p[39], p[40], p[41]), f3(p[45], p[46], p[47]));
  float*            q = out + (size_t)i * 8;
  q[0] = d.k2.x;
  q[1] = d.k2.y;
  q[2] = d.k2.z;
  q[3] = d.bsdf_over_pdf.x;
  q[4] = d.bsdf_over_pdf.y;
  q[5] = d.bsdf_over_pdf.z;
  q[6] = d.pdf;
  q[7] = (float)d.event_type;
}

// -------------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------------
}  // namespace

struct b200pt
{
  int          device = 0;
  cudaStream_t stream = nullptr;
  std::string  err;
  int          numSMs = 148;

  // scene
  std::vector<void*>  sceneAllocs;
  const void*         treeBase = nullptr;  // the trees' node + triangle arrays (one allocation) and their size: the L2 window
  size_t              treeBytes = 0;
  // opacity micromaps as handed over by b200pt_set_opacity_micromaps (host copies; consumed by the next b200pt_set_scene)
  struct OmmHost
  {
    std::vector<uint8_t>                  data;
    std::vector<b200pt_micromap_triangle> tris;
  };
  struct PrimOmmHost
  {
    uint32_t             prim = 0, micromap = 0, base = 0;
    bool                 hasIdx = false;
    std::vector<int32_t> idx;
  };
  std::vector<OmmHost>     omms;
  std::vector<PrimOmmHost> primOmms;
  uint32_t                 ommTriangles = 0;  // non-opaque triangles of the scene that got a micromap / special state
  DevScene            S{};
  bool                haveScene = false;
  bool                hasVolume = false;
  int                 bvhBuilder = 0;  // 0: host SAH builder (bvh.cpp), 1: device LBVH (lbvh.cuh); b200pt_set_bvh_builder
  double              bvhBuildMs = 0.0;  // wall time of the last scene's tree builds
  bool                leanShade = false;  // scene fits the FEAT_LEAN shade variant (scene_feature_detection analogue)
  uint32_t            featureMask = 0;
  uint64_t            nodeBytes = 0, triBytes = 0;
  uint32_t            numNodes = 0, numTris = 0;
  // writable views of the trees for b200pt_update_transforms (refit): [0] merged, [1] opaque-only, [2] non-opaque
  struct TreeDev
  {
    float*                                     nodes = nullptr;
    float*                                     tris = nullptr;   // the triangle array the tree indexes ([1] and [2] share one)
    uint2*                                     meta = nullptr;
    float4*                                    nodeBox = nullptr;  // 2 per node: world-space box (refit scratch)
    uint32_t                                   numNodes = 0, numTriSlots = 0;
    std::vector<std::pair<uint32_t, uint32_t>> levels;  // (first node, count) per depth: builders emit breadth first
  };
  TreeDev             tree[3];
  uint32_t            numSceneNodes = 0;
  b200pt_render_node* dNodesW = nullptr;  // == S.nodes, writable
  const DevPrim*      dPrimsW = nullptr;
  // animation feed (b200pt_set_animation / b200pt_animate): host copy of every primitive's device arrays + sizes, the writable
  // shade records, the uploaded static task inputs and the per-frame buffers (m_morphWeightsBuffer / m_jointMatricesBuffer /
  // m_normalMatricesBuffer of SceneAnimationVk, with per-task offsets)
  struct PrimHost
  {
    DevPrim  d{};
    uint32_t vertexCount = 0, triCount = 0, recBase = 0;
  };
  std::vector<PrimHost>     primHost;
  ShadeRec*                 dShadeRecsW = nullptr;
  std::vector<void*>        animAllocs;
  std::vector<MorphTaskDev> morphTasks;
  std::vector<SkinTaskDev>  skinTasks;
  std::vector<uint32_t>     morphPrim, skinPrim;  // renderPrimID per task
  float *                   dMorphWeights = nullptr, *dJointMats = nullptr, *dNormalMats = nullptr;
  size_t                    numMorphWeights = 0, numJoints = 0;
  // node hierarchy on the device (b200pt_set_node_hierarchy / b200pt_update_node_matrices)
  std::vector<void*>        graphAllocs;
  std::vector<uint32_t>     levelOffsets;
  uint32_t                  numGraphNodes = 0;
  int *                     dParents = nullptr, *dTopo = nullptr;
  float *                   dLocalMats = nullptr, *dWorldMats = nullptr, *dInstLocal = nullptr;
  RenderNodeMapping*        dMappings = nullptr;

  // env
  float4* dEnv = nullptr;
  uint2*  dEnvAccel = nullptr;
  bool    haveEnv = false;

  // framebuffer + path pool
  int                width = 0, height = 0, tileY0 = 0, tileRows = 0;
  int                bandRows = 0, bandWorld = 1, bandRank = 0;
  uint32_t           numPaths = 0;
  float4*            dAccumOwned = nullptr;
  float4*            dAccum = nullptr;
  bool               guides = false;      // b200pt_set_guide_outputs: the path pools carry guideA / guideN, dGuide is the eOptixAlbedoNormal image
  float4*            dGuide = nullptr;
  uchar4*            dTonemapped = nullptr;  // gBuffers[eImgTonemapped] of this tile (b200pt_tonemap), in poolAllocs
  uint32_t*          dTmHist = nullptr;      // 256-bin log2-luminance histogram + the exposure factor behind it (allocated with the handle)
  uint32_t*          dSelect = nullptr;  // frame-0 outputs (gltf_pathtrace.slang:610-616): object id per pixel ...
  float*             dNdcDepth = nullptr;  // ... and NDC depth of the first hit
  // Frames in flight (like the reference app's swapchain ring): every lane owns a stream, a path pool, queues and
  // counters; frame f runs its bounces on lane f % numLanes and only k_accumulate runs on the main stream, in
  // frame order.  The latency-bound tail of frame f (a few deep paths) overlaps the wide first bounces of f+1.
  struct Lane
  {
    cudaStream_t stream = nullptr;
    PathState    P{};
    uint32_t*    dQ[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // trace ping/pong, post, shadow, alpha, continuation
    uint32_t*    dCounters = nullptr;
    uint32_t*    hCount = nullptr;   // pinned
    cudaEvent_t  done = nullptr;     // lane stream: all bounces of the lane's frame enqueued before it
    cudaEvent_t  freed = nullptr;    // main stream: k_accumulate has consumed the lane's pixSum
    bool         busy = false;       // `freed` has been recorded at least once since the pool was (re)built
  };
  static constexpr int kMaxLanes = 8;
  Lane               lanes[kMaxLanes];
  // frame batching (b200pt_set_frame_batch): up to `batch` consecutive frames of a static camera are collected and run as one
  // wavefront of batch x pixels paths (a multi-GPU tile is 1/N of the frame: batching N frames gives its kernels the size of a
  // single-GPU frame and divides the launches per frame by N)
  int                   batch = 1;
  int                   pendingCount = 0;
  b200pt_frame_info     pendingFi{};
  b200pt_push_constant  pendingPc{};  // the FIRST pending frame's constants
  int                numLanes = 4;   // measured on B200 (1080p bench): 1 -> 310, 2 -> 366, 3 -> 378 Mray/s (first version); 3 -> 599, 4 -> 617, 6 -> 622 (now)
  uint64_t           frameSerial = 0;
  int                lastLane = -1;
  cudaEvent_t        readDone[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  std::vector<void*> poolAllocs;
  // scratch pool of the ray-level API (b200pt_trace_closest / b200pt_trace_shadow run the production kernels on it)
  PathState          rayP{};
  uint32_t*          rayQ[3] = {nullptr, nullptr, nullptr};  // rays, any-hit, continuation
  uint32_t*          rayCounters = nullptr;                  // 8 words
  uint32_t           rayCapacity = 0;
  std::vector<void*> rayAllocs;
  DevStats*          dStats = nullptr;
  float*             dLutSrgb = nullptr;

  // stats / profiling: CUDA-event pairs recorded around every launch on the handle's stream and
  // resolved lazily (no host sync inside a frame)
  struct EvRec
  {
    cudaEvent_t a, b;
    int         cat;
    int         lane;  // timeline: stream the launch went to (-1 main)
    uint64_t    frame;
  };
  bool               profiling = false;
  // B200PT_TIMELINE=<file>: event pairs around every launch WITHOUT serialising the frames in flight; flushEvents appends
  // "frame,lane,stage,start_ms,end_ms" rows (times relative to tlBase) -- the per-rank timeline of a real run
  FILE*              timeline = nullptr;
  cudaEvent_t        tlBase = nullptr;
  std::vector<EvRec> evPool;
  size_t             evUsed = 0;
  double             msCat[6] = {0, 0, 0, 0, 0, 0};  // 0 k_trace, 1 k_shade, 2 k_shadow, 3 other, 4 k_alpha, 5 k_resolve
  uint64_t           launchesCat[6] = {0, 0, 0, 0, 0, 0};
  uint64_t           kernelLaunches = 0;
};

namespace {

#define CK(call)                                                                                                                            \
  do                                                                                                                                        \
  {                                                                                                                                         \
    cudaError_t e__ = (call);                                                                                                               \
    if(e__ != cudaSuccess)                                                                                                                  \
    {                                                                                                                                       \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e__);                                                                         \
      return B200PT_E_CUDA;                                                                                                                 \
    }                                                                                                                                       \
  } while(0)

template <typename T>
int upload(b200pt* h, std::vector<void*>& owner, const T* src, size_t count, T** out)
{
  *out = nullptr;
  const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
  void*        d = nullptr;
  CK(cudaMalloc(&d, bytes));
  owner.push_back(d);
  if(count)
    CK(cudaMemcpyAsync(d, src, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  else
    CK(cudaMemsetAsync(d, 0, bytes, h->stream));
  *out = (T*)d;
  return 0;
}

// the SoA arrays of one path pool (device_scene.cuh: PathState) for n paths
int allocPathState(b200pt* h, std::vector<void*>& owner, size_t n, PathState& P)
{
  P = PathState{};
  float4** arrays[] = {&P.rayO, &P.rayD, &P.hit, &P.thr, &P.rad, &P.misc, reinterpret_cast<float4**>(&P.medium), &P.pixSum, &P.shO, &P.shD, &P.shC, &P.firstHit};
  for(float4** a : arrays)
  {
    void* d = nullptr;
    if(cudaMalloc(&d, std::max<size_t>(n, 1) * 16) != cudaSuccess)
    {
      cudaGetLastError();
      h->err = "path pool: out of device memory";
      return B200PT_E_NOMEM;
    }
    owner.push_back(d);
    *a = reinterpret_cast<float4*>(d);
  }
  for(int k = 0; k < kCand; k++)
  {
    void* d = nullptr;
    if(cudaMalloc(&d, std::max<size_t>(n, 1) * 16) != cudaSuccess)
    {
      cudaGetLastError();
      h->err = "path pool: out of device memory";
      return B200PT_E_NOMEM;
    }
    owner.push_back(d);
    P.cand[k] = reinterpret_cast<float4*>(d);
  }
  void* d = nullptr;
  if(cudaMalloc(&d, std::max<size_t>(n, 1) * sizeof(uint2)) != cudaSuccess)
  {
    cudaGetLastError();
    h->err = "path pool: out of device memory";
    return B200PT_E_NOMEM;
  }
  owner.push_back(d);
  P.candInfo = reinterpret_cast<uint2*>(d);
  if(h->guides)
    for(float4** a : {&P.guideA, &P.guideN})
    {
      void* g = nullptr;
      if(cudaMalloc(&g, std::max<size_t>(n, 1) * 16) != cudaSuccess)
      {
        cudaGetLastError();
        h->err = "path pool: out of device memory";
        return B200PT_E_NOMEM;
      }
      owner.push_back(g);
      *a = reinterpret_cast<float4*>(g);
    }
  return B200PT_OK;
}

// Builds one compressed wide BVH over `m` of the scene's triangles ON THE DEVICE (lbvh.cuh) and brings it back in the host
// builder's format, so that everything downstream of the builders (uploads, record tables, refit levels) is shared.
// dInRec: 12 floats per global triangle in flatten order; dSubset: m global ids or nullptr.
int buildWideBvhGpu(b200pt* h, const float* dInRec, const uint32_t* dSubset, uint32_t m, uint32_t triBaseOffset, WideBvh& out)
{
  out = WideBvh();
  out.numTris = m;
  if(m == 0)
  {
    out.nodes.assign(20, 0.f);
    out.numNodes = 1;
    return B200PT_OK;
  }
  uint32_t M = 1;
  while(M < m)
    M <<= 1;
  std::vector<void*> tmp;
  auto               dalloc = [&](size_t bytes) -> void* {
    void* p = nullptr;
    if(cudaMalloc(&p, std::max<size_t>(bytes, 16)) != cudaSuccess)
    {
      cudaGetLastError();
      return nullptr;
    }
    tmp.push_back(p);
    return p;
  };
  auto cleanup = [&](int rc) {
    for(void* p : tmp)
      cudaFree(p);
    if(rc)
      h->err = "GPU BVH build failed (allocation or launch)";
    return rc;
  };
  LbvhWork W{};
  W.m = m;
  W.M = M;
  W.inRec = dInRec;
  W.subset = dSubset;
  W.triBaseOffset = triBaseOffset;
  W.primLo = (float4*)dalloc((size_t)m * 16);
  W.primHi = (float4*)dalloc((size_t)m * 16);
  W.keys = (unsigned long long*)dalloc((size_t)M * 8);
  W.left = (int*)dalloc((size_t)m * 4);
  W.right = (int*)dalloc((size_t)m * 4);
  W.parentI = (int*)dalloc((size_t)m * 4);
  W.parentL = (int*)dalloc((size_t)m * 4);
  W.first = (uint32_t*)dalloc((size_t)m * 4);
  W.last = (uint32_t*)dalloc((size_t)m * 4);
  W.boxLo = (float4*)dalloc((size_t)m * 16);
  W.boxHi = (float4*)dalloc((size_t)m * 16);
  W.visits = (uint32_t*)dalloc((size_t)m * 4);
  W.cbounds = (int*)dalloc(6 * 4);
  W.nodes = (float*)dalloc(((size_t)m + 1) * 80);
  W.tris = (float*)dalloc((size_t)m * 48);
  W.triMeta = (uint32_t*)dalloc((size_t)m * 8);
  W.counters = (uint32_t*)dalloc(4 * 4);
  int2* queue[2] = {(int2*)dalloc(((size_t)m + 1) * 8), (int2*)dalloc(((size_t)m + 1) * 8)};
  if(!W.primLo || !W.primHi || !W.keys || !W.left || !W.right || !W.parentI || !W.parentL || !W.first || !W.last || !W.boxLo || !W.boxHi || !W.visits || !W.cbounds
     || !W.nodes || !W.tris || !W.triMeta || !W.counters || !queue[0] || !queue[1])
    return cleanup(B200PT_E_NOMEM);
  cudaStream_t st = h->stream;
  const int    cbInit[6] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000};
  const uint32_t cnt0[4] = {1u, 0u, 0u, 0u};  // wide node 0 is the root
  bool         ok = cudaMemcpyAsync(W.cbounds, cbInit, sizeof(cbInit), cudaMemcpyHostToDevice, st) == cudaSuccess;
  ok = ok && cudaMemcpyAsync(W.counters, cnt0, sizeof(cnt0), cudaMemcpyHostToDevice, st) == cudaSuccess;
  ok = ok && cudaMemsetAsync(W.visits, 0, (size_t)m * 4, st) == cudaSuccess;
  ok = ok && cudaMemsetAsync(W.nodes, 0, ((size_t)m + 1) * 80, st) == cudaSuccess;
  if(!ok)
    return cleanup(B200PT_E_CUDA);
  const uint32_t gm = (m + 255) / 256, gM = (M + 255) / 256;
  k_lbvh_bounds<<<gm, 256, 0, st>>>(W);
  k_lbvh_morton<<<gM, 256, 0, st>>>(W);
  for(uint32_t k = 2; k <= M; k <<= 1)
    for(uint32_t j = k >> 1; j > 0; j >>= 1)
      k_lbvh_bitonic<<<gM, 256, 0, st>>>(W.keys, M, j, k);
  if(m >= 2)
  {
    k_lbvh_hierarchy<<<gm, 256, 0, st>>>(W);
    k_lbvh_fit<<<gm, 256, 0, st>>>(W);
  }
  h->kernelLaunches += 4;
  // collapse + emit, level by level
  const int2 rootEntry = make_int2(m >= 2 ? 0 : ~0, 0);
  if(cudaMemcpyAsync(queue[0], &rootEntry, sizeof(rootEntry), cudaMemcpyHostToDevice, st) != cudaSuccess)
    return cleanup(B200PT_E_CUDA);
  uint32_t count = 1, depth = 0;
  int      cur = 0;
  while(count)
  {
    const uint32_t zero = 0;
    if(cudaMemcpyAsync(&W.counters[2], &zero, 4, cudaMemcpyHostToDevice, st) != cudaSuccess)
      return cleanup(B200PT_E_CUDA);
    k_lbvh_emit<<<(count + 127) / 128, 128, 0, st>>>(W, queue[cur], count, queue[1 - cur]);
    h->kernelLaunches++;
    if(cudaMemcpyAsync(&count, &W.counters[2], 4, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
      return cleanup(B200PT_E_CUDA);
    cur = 1 - cur;
    depth++;
    if(depth > 64)
      return cleanup(B200PT_E_CUDA);
  }
  uint32_t cnt[2] = {0, 0};
  if(cudaMemcpy(cnt, W.counters, 8, cudaMemcpyDeviceToHost) != cudaSuccess || cnt[1] != m || cnt[0] == 0 || cnt[0] > m + 1)
    return cleanup(B200PT_E_CUDA);
  out.numNodes = cnt[0];
  out.maxDepth = depth;
  out.nodes.resize((size_t)cnt[0] * 20);
  out.tris.resize((size_t)m * 12);
  out.triMeta.resize((size_t)m * 2);
  if(cudaMemcpy(out.nodes.data(), W.nodes, out.nodes.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess
     || cudaMemcpy(out.tris.data(), W.tris, out.tris.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess
     || cudaMemcpy(out.triMeta.data(), W.triMeta, out.triMeta.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess)
    return cleanup(B200PT_E_CUDA);
  return cleanup(B200PT_OK);
}

void freeRayPool(b200pt* h)
{
  for(void* p : h->rayAllocs)
    cudaFree(p);
  h->rayAllocs.clear();
  h->rayCapacity = 0;
}

void freeAnimation(b200pt* h)
{
  for(void* p : h->animAllocs)
    cudaFree(p);
  h->animAllocs.clear();
  h->morphTasks.clear();
  h->skinTasks.clear();
  h->morphPrim.clear();
  h->skinPrim.clear();
  h->dMorphWeights = h->dJointMats = h->dNormalMats = nullptr;
  h->numMorphWeights = h->numJoints = 0;
}

void freeHierarchy(b200pt* h)
{
  for(void* p : h->graphAllocs)
    cudaFree(p);
  h->graphAllocs.clear();
  h->levelOffsets.clear();
  h->numGraphNodes = 0;
  h->dParents = h->dTopo = nullptr;
  h->dLocalMats = h->dWorldMats = h->dInstLocal = nullptr;
  h->dMappings = nullptr;
}

void freeScene(b200pt* h)
{
  freeAnimation(h);
  freeHierarchy(h);
  for(void* p : h->sceneAllocs)
    cudaFree(p);
  h->sceneAllocs.clear();
  h->primHost.clear();
  h->dShadeRecsW = nullptr;
  h->haveScene = false;
}

void syncAll(b200pt* h)
{
  for(int l = 0; l < b200pt::kMaxLanes; l++)
    if(h->lanes[l].stream)
      cudaStreamSynchronize(h->lanes[l].stream);
  cudaStreamSynchronize(h->stream);
}

void freePool(b200pt* h)
{
  for(int l = 0; l < b200pt::kMaxLanes; l++)
    h->lanes[l].busy = false;
  h->lastLane = -1;
  for(void* p : h->poolAllocs)
    cudaFree(p);
  h->poolAllocs.clear();
  h->dAccumOwned = nullptr;
  h->dAccum = nullptr;
  h->dSelect = nullptr;
  h->dNdcDepth = nullptr;
  h->dTonemapped = nullptr;
  h->dGuide = nullptr;
  h->numPaths = 0;
  for(int l = 0; l < b200pt::kMaxLanes; l++)
  {
    h->lanes[l].P = PathState{};
    for(int k = 0; k < 6; k++)
      h->lanes[l].dQ[k] = nullptr;
  }
}

void flushEvents(b200pt* h)
{
  if(h->evUsed == 0)
    return;
  syncAll(h);
  static const char* const kStage[6] = {"k_trace", "k_shade", "k_shadow", "other", "k_alpha", "k_resolve"};
  for(size_t i = 0; i < h->evUsed; i++)
  {
    float ms = 0.f;
    if(cudaEventElapsedTime(&ms, h->evPool[i].a, h->evPool[i].b) == cudaSuccess)
    {
      h->msCat[h->evPool[i].cat] += ms;
      h->launchesCat[h->evPool[i].cat]++;
    }
    if(h->timeline && h->tlBase)
    {
      float t0 = 0.f, t1 = 0.f;
      if(cudaEventElapsedTime(&t0, h->tlBase, h->evPool[i].a) == cudaSuccess && cudaEventElapsedTime(&t1, h->tlBase, h->evPool[i].b) == cudaSuccess)
        fprintf(h->timeline, "%llu,%d,%s,%.4f,%.4f\n", (unsigned long long)h->evPool[i].frame, h->evPool[i].lane, kStage[h->evPool[i].cat], t0, t1);
    }
  }
  if(h->timeline)
    fflush(h->timeline);
  h->evUsed = 0;
}

float srgbToLinear(float c) { return (c <= 0.04045f) ? c / 12.92f : powf((c + 0.055f) / 1.055f, 2.4f); }
float linearToSrgb(float c) { return (c <= 0.0031308f) ? c * 12.92f : 1.055f * powf(c, 1.0f / 2.4f) - 0.055f; }

// mip chain like the reference's vkCmdBlitImage(VK_FILTER_LINEAR) loop (src/gltf_scene_vk.cpp:1254-1332):
// every level is the linear-filtered half-size copy of the previous 8-bit level (sRGB images are
// filtered in linear light and re-encoded).
void downsample(const std::vector<uint8_t>& src, int w, int h, bool srgb, std::vector<uint8_t>& dst, int nw, int nh)
{
  dst.resize((size_t)nw * nh * 4);
  std::vector<float> lin((size_t)w * h * 4);
  float              lutL[256], lutS[256];
  for(int i = 0; i < 256; i++)
  {
    lutL[i] = (float)i / 255.0f;
    lutS[i] = srgbToLinear((float)i / 255.0f);
  }
  for(size_t i = 0; i < (size_t)w * h; i++)
    for(int c = 0; c < 4; c++)
      lin[i * 4 + c] = (srgb && c < 3) ? lutS[src[i * 4 + c]] : lutL[src[i * 4 + c]];
  for(int y = 0; y < nh; y++)
    for(int x = 0; x < nw; x++)
    {
      const float sx = (x + 0.5f) * (float)w / (float)nw - 0.5f;
      const float sy = (y + 0.5f) * (float)h / (float)nh - 0.5f;
      int         x0 = (int)floorf(sx), y0 = (int)floorf(sy);
      const float fx = sx - x0, fy = sy - y0;
      const int   x1 = std::min(x0 + 1, w - 1), y1 = std::min(y0 + 1, h - 1);
      x0 = std::max(x0, 0);
      y0 = std::max(y0, 0);
      for(int c = 0; c < 4; c++)
      {
        const float a = lin[((size_t)y0 * w + x0) * 4 + c], b = lin[((size_t)y0 * w + x1) * 4 + c];
        const float cc = lin[((size_t)y1 * w + x0) * 4 + c], d = lin[((size_t)y1 * w + x1) * 4 + c];
        float       v = (a * (1 - fx) + b * fx) * (1 - fy) + (cc * (1 - fx) + d * fx) * fy;
        if(srgb && c < 3)
          v = linearToSrgb(v);
        dst[((size_t)y * nw + x) * 4 + c] = (uint8_t)std::min(255.0f, std::max(0.0f, floorf(v * 255.0f + 0.5f)));
      }
    }
}

struct MipChain
{
  std::vector<std::vector<uint8_t>> level;
  std::vector<int>                  w, h;
};

void buildMipChain(const b200pt_texture& src, MipChain& mc)
{
  int w = src.width, hh = src.height;
  mc.level.emplace_back(src.rgba8, src.rgba8 + (size_t)w * hh * 4);
  mc.w.push_back(w);
  mc.h.push_back(hh);
  while(w > 1 || hh > 1)
  {
    const int            nw = std::max(1, w / 2), nh = std::max(1, hh / 2);
    std::vector<uint8_t> nxt;
    downsample(mc.level.back(), w, hh, src.srgb != 0, nxt, nw, nh);
    mc.level.push_back(std::move(nxt));
    mc.w.push_back(nw);
    mc.h.push_back(nh);
    w = nw;
    hh = nh;
  }
}

// texels of one mip chain in the device layout: level after level, each as row-major 4x4-texel tiles
// (levels narrower than 4 texels are padded; the padding is never addressed)
void packTiled(const MipChain& mc, std::vector<uint32_t>& texels, uint32_t levelOfs[16])
{
  for(size_t l = 0; l < mc.level.size() && l < 16; l++)
  {
    const int w = mc.w[l], hh = mc.h[l], tpr = (w + 3) >> 2, tpc = (hh + 3) >> 2;
    levelOfs[l] = (uint32_t)texels.size();
    texels.resize(texels.size() + (size_t)tpr * tpc * 16, 0u);
    uint32_t*       dst = texels.data() + levelOfs[l];
    const uint32_t* src = reinterpret_cast<const uint32_t*>(mc.level[l].data());
    for(int y = 0; y < hh; y++)
      for(int x = 0; x < w; x++)
        dst[(((size_t)(y >> 2) * tpr + (x >> 2)) << 4) + ((y & 3) << 2) + (x & 3)] = src[(size_t)y * w + x];
  }
}

void describeTexture(const b200pt_texture& src, const MipChain& mc, DevTex& dev)
{
  const int levels = (int)std::min<size_t>(mc.level.size(), 16);
  // sampler quirks kept from getSampler (src/gltf_scene_vk.cpp:909-947): the mip mode follows magFilter
  dev.w0 = src.width;
  dev.h0 = src.height;
  dev.maxLevel = (float)(levels - 1);
  dev.wrapS = src.wrapS;
  dev.wrapT = src.wrapT;
  dev.srgb = src.srgb ? 1 : 0;
  dev.magLinear = (src.magFilter != 9728) ? 1 : 0;
  dev.minLinear = (src.minFilter == 9728 || src.minFilter == 9984 || src.minFilter == 9986) ? 0 : 1;
  dev.mipLinear = (src.magFilter != 9728) ? 1 : 0;
}

int gridFor(const b200pt* h, int perSM) { return h->numSMs * perSM; }

}  // namespace
extern "C" {
static int launchFrames(b200pt_t* h, const b200pt_frame_info* fi, const b200pt_push_constant* pc, int count);
static int flushPending(b200pt_t* h);
}
namespace {

// device-side error flags (DevStats::errorFlags) -> error code; the flag stays set until b200pt_reset_stats
int checkDeviceErrors(b200pt* h)
{
  unsigned long long flags = 0;
  if(cudaMemcpy(&flags, &h->dStats->errorFlags, sizeof(flags), cudaMemcpyDeviceToHost) != cudaSuccess)
  {
    h->err = "reading the device error flags failed";
    return B200PT_E_CUDA;
  }
  if(flags & 1ull)
  {
    h->err = "a traversal stack overflowed: the BVH is deeper than the kernels' stack, results are incomplete";
    return B200PT_E_DEVICE;
  }
  return B200PT_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int b200pt_abi_version(void) { return B200PT_ABI_VERSION; }

int b200pt_create(b200pt_t** out, int cuda_device)
{
  if(!out)
    return B200PT_E_INVALID;
  *out = nullptr;
  int n = 0;
  if(cudaGetDeviceCount(&n) != cudaSuccess || cuda_device < 0 || cuda_device >= n)
    return B200PT_E_CUDA;
  b200pt* h = new b200pt();
  h->device = cuda_device;
  if(cudaSetDevice(cuda_device) != cudaSuccess || cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
  {
    delete h;
    return B200PT_E_CUDA;
  }
  bool ok = true;
  auto need = [&](cudaError_t e) { ok = ok && (e == cudaSuccess); };
  cudaDeviceProp prop{};
  need(cudaGetDeviceProperties(&prop, cuda_device));
  h->numSMs = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
  need(cudaMalloc((void**)&h->dStats, sizeof(DevStats)));
  if(ok)
    need(cudaMemset(h->dStats, 0, sizeof(DevStats)));
  if(const char* e = getenv("B200PT_FRAMES_IN_FLIGHT"))
    h->numLanes = std::min(std::max(atoi(e), 1), (int)b200pt::kMaxLanes);
  if(const char* e = getenv("B200PT_TIMELINE"))
  {
    // one file per process (ranks of a multi-GPU run append their pid)
    const std::string path = std::string(e) + "." + std::to_string((long long)getpid());
    h->timeline = fopen(path.c_str(), "w");
    if(h->timeline)
    {
      fprintf(h->timeline, "frame,lane,stage,start_ms,end_ms\n");
      need(cudaEventCreate(&h->tlBase));
      need(cudaEventRecord(h->tlBase, h->stream));
      h->evPool.resize(16384);
      for(auto& ev : h->evPool)
      {
        need(cudaEventCreate(&ev.a));
        need(cudaEventCreate(&ev.b));
        ev.cat = 3;
      }
    }
  }
  for(int l = 0; l < b200pt::kMaxLanes; l++)
  {
    b200pt::Lane& L = h->lanes[l];
    need(cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
    need(cudaEventCreateWithFlags(&L.done, cudaEventDisableTiming));
    need(cudaEventCreateWithFlags(&L.freed, cudaEventDisableTiming));
    need(cudaMalloc((void**)&L.dCounters, sizeof(uint32_t) * kCounterArrays * kMaxIters));
    need(cudaMallocHost((void**)&L.hCount, sizeof(uint32_t) * 4));
  }
  {
    // [0..255]: sRGB decode; [256..511]: i / 255 (the UNORM decode, tabulated so that texel fetches do no divisions;
    // same IEEE quotient the kernel's own `(float)i / 255.0f` would produce)
    float lutS[512];
    for(int i = 0; i < 256; i++)
    {
      lutS[i] = srgbToLinear((float)i / 255.0f);
      lutS[256 + i] = (float)i / 255.0f;
    }
    need(cudaMalloc((void**)&h->dLutSrgb, sizeof(lutS)));
    need(cudaMalloc((void**)&h->dTmHist, (kTmBins + 1) * sizeof(uint32_t)));  // histogram + the exposure factor (a float in the last word)
    if(ok)
      need(cudaMemcpy(h->dLutSrgb, lutS, sizeof(lutS), cudaMemcpyHostToDevice));
  }
  if(!ok)
  {
    cudaGetLastError();  // clear the sticky-free error state for the next attempt
    b200pt_destroy(h);
    return B200PT_E_CUDA;
  }
  *out = h;
  return B200PT_OK;
}

void b200pt_destroy(b200pt_t* h)
{
  if(!h)
    return;
  cudaSetDevice(h->device);
  syncAll(h);
  flushEvents(h);  // (writes the tail of a B200PT_TIMELINE dump; needs the lane streams alive)
  freeScene(h);
  freePool(h);
  freeRayPool(h);
  for(int k = 0; k < 8; k++)
    if(h->readDone[k])
      cudaEventDestroy(h->readDone[k]);
  for(int l = 0; l < b200pt::kMaxLanes; l++)
  {
    b200pt::Lane& L = h->lanes[l];
    cudaFree(L.dCounters);
    if(L.hCount)
      cudaFreeHost(L.hCount);
    if(L.done)
      cudaEventDestroy(L.done);
    if(L.freed)
      cudaEventDestroy(L.freed);
    if(L.stream)
      cudaStreamDestroy(L.stream);
  }
  if(h->dEnv)
    cudaFree(h->dEnv);
  if(h->dEnvAccel)
    cudaFree(h->dEnvAccel);
  cudaFree(h->dStats);
  cudaFree(h->dLutSrgb);
  cudaFree(h->dTmHist);
  for(auto& e : h->evPool)
  {
    cudaEventDestroy(e.a);
    cudaEventDestroy(e.b);
  }
  if(h->tlBase)
    cudaEventDestroy(h->tlBase);
  if(h->timeline)
    fclose(h->timeline);
  cudaStreamDestroy(h->stream);
  delete h;
}

const char* b200pt_last_error(const b200pt_t* h) { return h ? h->err.c_str() : "null handle"; }

void* b200pt_stream(b200pt_t* h) { return h ? (void*)h->stream : nullptr; }

int b200pt_set_scene(b200pt_t* h, const b200pt_scene_desc* s)
{
  if(!h || !s || s->numMaterials == 0 || (s->numRenderNodes && (!s->renderNodes || !s->renderPrimitives)))
  {
    if(h)
      h->err = "b200pt_set_scene: invalid scene description";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  freeScene(h);
  DevScene& S = h->S;
  const int envW0 = S.envW, envH0 = S.envH;
  S = DevScene{};
  S.envRgba = h->dEnv;
  S.envAccel = h->dEnvAccel;
  S.envW = envW0;
  S.envH = envH0;
  S.lutSrgb = h->dLutSrgb;

  // --- AoS tables: same bytes as the reference SSBOs ---
  b200pt_render_node*    dNodes;
  b200pt_shade_material* dMats;
  b200pt_texture_info*   dTi;
  b200pt_light*          dLights;
  int                    rc;
  if((rc = upload(h, h->sceneAllocs, s->renderNodes, s->numRenderNodes, &dNodes)))
    return rc;
  if((rc = upload(h, h->sceneAllocs, s->materials, s->numMaterials, &dMats)))
    return rc;
  if((rc = upload(h, h->sceneAllocs, s->textureInfos, s->numTextureInfos, &dTi)))
    return rc;
  if((rc = upload(h, h->sceneAllocs, s->lights, s->numLights, &dLights)))
    return rc;
  // which KHR_materials_* features do the scene's materials use (reference: src/scene_feature_detection.cpp)
  {
    uint32_t feat = s->numLights ? FEAT_LIGHTS : 0u;
    for(uint32_t i = 0; i < s->numMaterials; i++)
    {
      const b200pt_shade_material& m = s->materials[i];
      // the 22 texture slots index GltfTextureInfo[] (0 = none, shaders/gltf_scene_io.h.slang:196-219)
      const uint16_t* slots = &m.pbrBaseColorTexture;
      for(int k = 0; k < 22; k++)
        if(slots[k] != 0 && slots[k] >= s->numTextureInfos)
        {
          h->err = "b200pt_set_scene: material texture slot beyond numTextureInfos";
          return B200PT_E_INVALID;
        }
      if(m.retroreflectionFactor > 0.0f)
      {
        h->err = "b200pt_set_scene: KHR_materials_retroreflection is not built (its lobe lives in nvshaders, external to the reference tree)";
        return B200PT_E_UNSUPPORTED;
      }
      if(m.transmissionFactor > 0.0f || m.transmissionTexture)
        feat |= FEAT_TRANSMISSION;
      if(m.thicknessFactor > 0.0f || m.thicknessTexture || m.multiscatterColorFactor[0] > 0.0f || m.multiscatterColorFactor[1] > 0.0f || m.multiscatterColorFactor[2] > 0.0f)
        feat |= FEAT_VOLUME;
      if(m.diffuseTransmissionFactor > 0.0f || m.diffuseTransmissionTexture)
        feat |= FEAT_DIFFUSE_TRANSMISSION;
      if(m.clearcoatFactor > 0.0f)
        feat |= FEAT_CLEARCOAT;
      if(m.sheenColorFactor[0] != 0.0f || m.sheenColorFactor[1] != 0.0f || m.sheenColorFactor[2] != 0.0f)
        feat |= FEAT_SHEEN;
      if(m.iridescenceFactor > 0.0f)
        feat |= FEAT_IRIDESCENCE;
      if(m.anisotropyStrength > 0.0f)
        feat |= FEAT_ANISOTROPY;
      if(m.pbrModel == 1)
        feat |= FEAT_SPECGLOSS;
    }
    h->featureMask = feat;
    h->leanShade = (feat & ~(uint32_t)FEAT_LEAN) == 0;
  }
  S.nodes = dNodes;
  S.mats = dMats;
  S.texInfos = dTi;
  S.lights = dLights;
  S.numLights = (int)s->numLights;

  // --- vertex data: separate attribute arrays per primitive, as SceneVk::createVertexBuffers ---
  std::vector<DevPrim> prims(s->numRenderPrimitives);
  for(uint32_t i = 0; i < s->numRenderPrimitives; i++)
  {
    const b200pt_render_primitive& p = s->renderPrimitives[i];
    DevPrim&                       d = prims[i];
    uint32_t*                      di;
    float*                         df;
    if((rc = upload(h, h->sceneAllocs, p.indices, (size_t)p.triangleCount * 3, &di)))
      return rc;
    d.idx = di;
    if((rc = upload(h, h->sceneAllocs, p.positions, (size_t)p.vertexCount * 3, &df)))
      return rc;
    d.pos = df;
    d.nrm = d.tan = d.uv0 = d.uv1 = nullptr;
    d.col = nullptr;
    if(p.normals)
    {
      if((rc = upload(h, h->sceneAllocs, p.normals, (size_t)p.vertexCount * 3, &df)))
        return rc;
      d.nrm = df;
    }
    if(p.tangents)
    {
      if((rc = upload(h, h->sceneAllocs, p.tangents, (size_t)p.vertexCount * 4, &df)))
        return rc;
      d.tan = df;
    }
    if(p.texCoords[0])
    {
      if((rc = upload(h, h->sceneAllocs, p.texCoords[0], (size_t)p.vertexCount * 2, &df)))
        return rc;
      d.uv0 = df;
    }
    if(p.texCoords[1])
    {
      if((rc = upload(h, h->sceneAllocs, p.texCoords[1], (size_t)p.vertexCount * 2, &df)))
        return rc;
      d.uv1 = df;
    }
    if(p.colors)
    {
      if((rc = upload(h, h->sceneAllocs, p.colors, (size_t)p.vertexCount, &di)))
        return rc;
      d.col = di;
    }
  }
  DevPrim* dPrims;
  if((rc = upload(h, h->sceneAllocs, prims.data(), prims.size(), &dPrims)))
    return rc;
  S.prims = dPrims;
  h->primHost.resize(s->numRenderPrimitives);
  for(uint32_t i = 0; i < s->numRenderPrimitives; i++)
  {
    h->primHost[i].d = prims[i];
    h->primHost[i].vertexCount = s->renderPrimitives[i].vertexCount;
    h->primHost[i].triCount = s->renderPrimitives[i].triangleCount;
  }

  // --- textures ---
  std::vector<DevTex> devTex(s->numTextures);
  std::vector<const uchar4*> texLevel0(s->numTextures, nullptr);  // level-0 texels (device), for the alpha-triangle records
  {
    for(uint32_t i = 0; i < s->numTextures; i++)
      if(s->textures[i].width <= 0 || s->textures[i].height <= 0 || !s->textures[i].rgba8)
      {
        h->err = "texture without pixels";
        return B200PT_E_INVALID;
      }
    std::vector<MipChain>    chains(s->numTextures);
    std::atomic<uint32_t>    nextTex{0};
    std::vector<std::thread> workers;
    auto                     job = [&]() {
      for(uint32_t i = nextTex.fetch_add(1); i < s->numTextures; i = nextTex.fetch_add(1))
        buildMipChain(s->textures[i], chains[i]);
    };
    const unsigned nt = std::max(1u, std::min(std::thread::hardware_concurrency(), s->numTextures));
    for(unsigned t = 1; t < nt; t++)
      workers.emplace_back(job);
    job();
    for(auto& t : workers)
      t.join();
    // one allocation for all texels, one table of level offsets
    std::vector<uint32_t> levelOfs((size_t)s->numTextures * 16, 0u);
    std::vector<size_t>   texBase(s->numTextures, 0);
    size_t                total = 0;
    std::vector<std::vector<uint32_t>> packed(s->numTextures);
    {
      std::atomic<uint32_t>    nextPack{0};
      std::vector<std::thread> packers;
      auto                     pjob = [&]() {
        for(uint32_t i = nextPack.fetch_add(1); i < s->numTextures; i = nextPack.fetch_add(1))
          packTiled(chains[i], packed[i], &levelOfs[(size_t)i * 16]);
      };
      for(unsigned t = 1; t < nt; t++)
        packers.emplace_back(pjob);
      pjob();
      for(auto& t : packers)
        t.join();
    }
    for(uint32_t i = 0; i < s->numTextures; i++)
    {
      texBase[i] = total;
      total += packed[i].size();
    }
    uint32_t* dTexels = nullptr;
    uint32_t* dLevelOfs = nullptr;
    CK(cudaMalloc((void**)&dTexels, std::max<size_t>(total, 1) * sizeof(uint32_t)));
    h->sceneAllocs.push_back(dTexels);
    for(uint32_t i = 0; i < s->numTextures; i++)
      CK(cudaMemcpy(dTexels + texBase[i], packed[i].data(), packed[i].size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    if((rc = upload(h, h->sceneAllocs, levelOfs.data(), levelOfs.size(), &dLevelOfs)))
      return rc;
    for(uint32_t i = 0; i < s->numTextures; i++)
    {
      describeTexture(s->textures[i], chains[i], devTex[i]);
      devTex[i].texels = reinterpret_cast<const uchar4*>(dTexels + texBase[i]);
      texLevel0[i] = devTex[i].texels + levelOfs[(size_t)i * 16];
      devTex[i].levelOfs = dLevelOfs + (size_t)i * 16;
    }
  }
  DevTex* dTex;
  if((rc = upload(h, h->sceneAllocs, devTex.data(), devTex.size(), &dTex)))
    return rc;
  S.textures = dTex;
  S.numTextures = (int)s->numTextures;

  // --- flatten instances to world space + build the wide BVH (TLAS/BLAS replacement) ---
  std::vector<FlatTri> flat;
  h->hasVolume = false;
  for(uint32_t n = 0; n < s->numRenderNodes; n++)
  {
    if(s->renderNodeVisible && !s->renderNodeVisible[n])
      continue;
    const b200pt_render_node& node = s->renderNodes[n];
    if(node.renderPrimID < 0 || (uint32_t)node.renderPrimID >= s->numRenderPrimitives)
    {
      h->err = "render node references a missing primitive";
      return B200PT_E_INVALID;
    }
    const b200pt_render_primitive& p = s->renderPrimitives[node.renderPrimID];
    if(node.materialID >= (int)s->numMaterials)
    {
      h->err = "render node references a missing material";
      return B200PT_E_INVALID;
    }
    const b200pt_shade_material&   m = s->materials[(uint32_t)std::max(0, node.materialID)];
    uint32_t                       flags = 0;
    if(m.transmissionFactor == 0.0f && m.alphaMode == 0 && m.diffuseTransmissionFactor == 0.0f)
      flags |= TRI_OPAQUE;
    if(m.doubleSided == 1 || m.thicknessFactor > 0.0f || m.transmissionFactor > 0.0f)
      flags |= TRI_NOCULL;
    // a path can take more than maxDepth wavefront iterations exactly when k_shade can scatter inside a medium: that
    // is gated on the medium's scatter coefficient (multiscatterColorFactor), not on thickness (makeVolumeMedium runs on
    // every transmission event, pathtrace_functions.h.slang:118-140, 605-672)
    if((m.transmissionFactor > 0.0f || m.transmissionTexture || m.diffuseTransmissionFactor > 0.0f || m.diffuseTransmissionTexture)
       && (m.multiscatterColorFactor[0] > 0.0f || m.multiscatterColorFactor[1] > 0.0f || m.multiscatterColorFactor[2] > 0.0f))
      h->hasVolume = true;
    const float* a = node.objectToWorld;
    const float  det = a[0] * (a[5] * a[10] - a[9] * a[6]) - a[4] * (a[1] * a[10] - a[9] * a[2]) + a[8] * (a[1] * a[6] - a[5] * a[2]);
    const bool   mirrored = det < 0.0f;
    for(uint32_t t = 0; t < p.triangleCount; t++)
    {
      float3 v[3];
      for(int k = 0; k < 3; k++)
      {
        const uint32_t vi = p.indices[t * 3 + k];
        if(vi >= p.vertexCount)
        {
          h->err = "b200pt_set_scene: index beyond the primitive's vertex count";
          return B200PT_E_INVALID;
        }
        v[k] = xfPoint(a, f3(p.positions[vi * 3], p.positions[vi * 3 + 1], p.positions[vi * 3 + 2]));
      }
      FlatTri T;
      T.rnode = n;
      T.prim = t;
      T.flags = flags;
      if(mirrored)
      {
        std::swap(v[1], v[2]);
        T.flags |= TRI_FLIPPED;
      }
      const float3 e1 = v[1] - v[0], e2 = v[2] - v[0];
      T.v0[0] = v[0].x, T.v0[1] = v[0].y, T.v0[2] = v[0].z;
      T.e1[0] = e1.x, T.e1[1] = e1.y, T.e1[2] = e1.z;
      T.e2[0] = e2.x, T.e2[1] = e2.y, T.e2[2] = e2.z;
      flat.push_back(T);
    }
  }
  // ONE tree over every triangle (opaque and any-hit geometry alike: the per-triangle TRI_OPAQUE flag decides what a
  // geometric hit means, traverse.cuh); the global triangle id (flatten order) is the tie-break key
  std::vector<uint32_t> gids(flat.size());
  bool                  anyNonOpaque = false;
  for(uint32_t i = 0; i < (uint32_t)flat.size(); i++)
  {
    gids[i] = i;
    anyNonOpaque = anyNonOpaque || !(flat[i].flags & TRI_OPAQUE);
  }
  // closest-hit rays walk the merged tree; shadow rays walk an opaque-only tree first (any hit ends the query, occluded
  // rays never meet the foliage boxes) and the non-opaque tree after it (traverse.cuh).  The three builds run in parallel.
  WideBvh bvh, bvhO, bvhA;
  {
    std::vector<FlatTri>  flatO, flatA;
    std::vector<uint32_t> gidO, gidA;
    if(anyNonOpaque)
      for(uint32_t i = 0; i < (uint32_t)flat.size(); i++)
      {
        if(flat[i].flags & TRI_OPAQUE)
        {
          flatO.push_back(flat[i]);
          gidO.push_back(i);
        }
        else
        {
          flatA.push_back(flat[i]);
          gidA.push_back(i);
        }
      }
    const auto tBuild0 = std::chrono::steady_clock::now();
    if(h->bvhBuilder == 1)
    {
      // device LBVH: the flattened records go up once (flatten order = global id order), the subsets as id lists
      std::vector<float> rec(flat.size() * 12);
      for(size_t i = 0; i < flat.size(); i++)
      {
        const FlatTri& T = flat[i];
        float*         R = &rec[i * 12];
        const uint32_t w0 = T.rnode | (T.flags << 28), prim = T.prim, gid = (uint32_t)i;
        memcpy(R, T.v0, 12);
        memcpy(R + 3, &w0, 4);
        memcpy(R + 4, T.e1, 12);
        memcpy(R + 7, &prim, 4);
        memcpy(R + 8, T.e2, 12);
        memcpy(R + 11, &gid, 4);
      }
      float *   dRec = nullptr;
      uint32_t *dO = nullptr, *dA = nullptr;
      std::vector<void*> tmpAllocs;
      if((rc = upload(h, tmpAllocs, rec.data(), rec.size(), &dRec)) == 0 && anyNonOpaque)
      {
        rc = upload(h, tmpAllocs, gidO.data(), gidO.size(), &dO);
        if(!rc)
          rc = upload(h, tmpAllocs, gidA.data(), gidA.size(), &dA);
      }
      if(!rc)
        rc = buildWideBvhGpu(h, dRec, nullptr, (uint32_t)flat.size(), 0u, bvh);
      if(!rc && anyNonOpaque)
      {
        rc = buildWideBvhGpu(h, dRec, dO, (uint32_t)gidO.size(), 0u, bvhO);
        if(!rc)
          rc = buildWideBvhGpu(h, dRec, dA, (uint32_t)gidA.size(), (uint32_t)gidO.size(), bvhA);
      }
      cudaStreamSynchronize(h->stream);
      for(void* p : tmpAllocs)
        cudaFree(p);
      if(rc)
        return rc;
    }
    else
    {
      std::thread tO, tA;
      if(anyNonOpaque)
      {
        tO = std::thread([&] { buildWideBvh(flatO, gidO, 0u, bvhO); });
        tA = std::thread([&] { buildWideBvh(flatA, gidA, (uint32_t)flatO.size(), bvhA); });
      }
      buildWideBvh(flat, gids, 0u, bvh);
      if(anyNonOpaque)
      {
        tO.join();
        tA.join();
      }
    }
    h->bvhBuildMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tBuild0).count();
  }
  // The node and triangle arrays of all three trees live in ONE allocation, so that a single L2 access-policy window can pin them
  // (setTreeWindow below): the walks re-read these few tens of MB all the time while every bounce streams GBs of path state past them.
  std::vector<float> trisS, packed;
  size_t             offTris = 0, offNodesO = 0, offNodesA = 0, offTrisS = 0;
  {
    auto place = [&](const std::vector<float>& v) {
      const size_t at = packed.size();
      packed.insert(packed.end(), v.begin(), v.end());
      packed.resize((packed.size() + 31) & ~(size_t)31, 0.0f);  // 128-byte granules
      return at;
    };
    place(bvh.nodes);
    offTris = place(bvh.tris);
    if(anyNonOpaque)
    {
      trisS = bvhO.tris;
      trisS.insert(trisS.end(), bvhA.tris.begin(), bvhA.tris.end());
      offNodesO = place(bvhO.nodes);
      offNodesA = place(bvhA.nodes);
      offTrisS = place(trisS);
    }
  }
  float *   dPacked, *dBvhNodes, *dTris;
  uint32_t* dMeta;
  if((rc = upload(h, h->sceneAllocs, packed.data(), packed.size(), &dPacked)))
    return rc;
  dBvhNodes = dPacked;
  dTris = dPacked + offTris;
  h->treeBase = dPacked;
  h->treeBytes = packed.size() * sizeof(float);
  if((rc = upload(h, h->sceneAllocs, bvh.triMeta.data(), bvh.triMeta.size(), &dMeta)))
    return rc;
  S.bvh.nodes = reinterpret_cast<const float4*>(dBvhNodes);
  S.bvh.tris = reinterpret_cast<const float4*>(dTris);
  S.bvh.ommRef = nullptr;
  S.bvh.ommData = nullptr;
  S.hasAlpha = anyNonOpaque ? 1 : 0;
  S.triMeta = reinterpret_cast<const uint2*>(dMeta);
  S.bvhO = S.bvh;
  S.bvhA = S.bvh;
  S.triMetaS = S.triMeta;
  // breadth-first level ranges of a tree (the builder emits level by level, so every level is one contiguous index range)
  auto levelsOf = [](const WideBvh& t) {
    std::vector<std::pair<uint32_t, uint32_t>> lv;
    uint32_t                                   first = 0, count = 1;
    while(count)
    {
      lv.push_back({first, count});
      uint32_t next = 0;
      for(uint32_t n = first; n < first + count; n++)
      {
        uint32_t w;
        memcpy(&w, &t.nodes[(size_t)n * 20 + 3], 4);
        next += (uint32_t)__builtin_popcount(w >> 24);
      }
      first += count;
      count = next;
    }
    return lv;
  };
  for(auto& t : h->tree)
    t = b200pt::TreeDev();
  h->tree[0].nodes = dBvhNodes;
  h->tree[0].tris = dTris;
  h->tree[0].meta = reinterpret_cast<uint2*>(dMeta);
  h->tree[0].numNodes = bvh.numNodes;
  h->tree[0].numTriSlots = bvh.numTris;
  h->tree[0].levels = levelsOf(bvh);
  uint64_t splitNodeBytes = 0, splitTriBytes = 0;
  if(anyNonOpaque)
  {
    std::vector<uint32_t> metaS(bvhO.triMeta);
    metaS.insert(metaS.end(), bvhA.triMeta.begin(), bvhA.triMeta.end());
    float *   dNodesO = dPacked + offNodesO, *dNodesA = dPacked + offNodesA, *dTrisS = dPacked + offTrisS;
    uint32_t* dMetaS;
    if((rc = upload(h, h->sceneAllocs, metaS.data(), metaS.size(), &dMetaS)))
      return rc;
    S.bvhO.nodes = reinterpret_cast<const float4*>(dNodesO);
    S.bvhO.tris = reinterpret_cast<const float4*>(dTrisS);
    S.bvhA.nodes = reinterpret_cast<const float4*>(dNodesA);
    S.bvhA.tris = reinterpret_cast<const float4*>(dTrisS);
    S.triMetaS = reinterpret_cast<const uint2*>(dMetaS);
    splitNodeBytes = (bvhO.nodes.size() + bvhA.nodes.size()) * sizeof(float);
    splitTriBytes = trisS.size() * sizeof(float);
    h->tree[1].nodes = dNodesO;
    h->tree[1].tris = dTrisS;
    h->tree[1].meta = reinterpret_cast<uint2*>(dMetaS);
    h->tree[1].numNodes = bvhO.numNodes;
    h->tree[1].numTriSlots = bvhO.numTris + bvhA.numTris;  // the shared array is refitted once, through this entry
    h->tree[1].levels = levelsOf(bvhO);
    h->tree[2].nodes = dNodesA;
    h->tree[2].tris = dTrisS;
    h->tree[2].meta = nullptr;
    h->tree[2].numNodes = bvhA.numNodes;
    h->tree[2].numTriSlots = 0;
    h->tree[2].levels = levelsOf(bvhA);
  }
  for(auto& t : h->tree)
    if(t.nodes)
    {
      CK(cudaMalloc((void**)&t.nodeBox, (size_t)std::max(t.numNodes, 1u) * 2 * sizeof(float4)));
      h->sceneAllocs.push_back(t.nodeBox);
    }
  h->numSceneNodes = s->numRenderNodes;
  h->dNodesW = dNodes;
  h->dPrimsW = dPrims;
  // ---- per-triangle attribute records for getHitState (device_scene.cuh: ShadeRec), per render primitive ----
  {
    std::vector<uint32_t> recBase(s->numRenderPrimitives, 0);
    size_t                total = 0;
    for(uint32_t i = 0; i < s->numRenderPrimitives; i++)
    {
      recBase[i] = (uint32_t)total;
      total += s->renderPrimitives[i].triangleCount;
    }
    std::vector<ShadeRec> recs(total);
    for(uint32_t i = 0; i < s->numRenderPrimitives; i++)
    {
      const b200pt_render_primitive& p = s->renderPrimitives[i];
      for(uint32_t t = 0; t < p.triangleCount; t++)
      {
        ShadeRec& r = recs[recBase[i] + t];
        float*    f = reinterpret_cast<float*>(&r);  // 48 floats, layout: device_scene.cuh ShadeRec
        memset(f, 0, sizeof(ShadeRec));
        const uint32_t flags = (p.normals ? 1u : 0u) | (p.texCoords[0] ? 2u : 0u) | (p.texCoords[1] ? 4u : 0u) | (p.colors ? 8u : 0u) | (p.tangents ? 16u : 0u);
        memcpy(&f[3], &flags, 4);
        uint32_t vi[3];
        for(int c = 0; c < 3; c++)
        {
          vi[c] = p.indices[t * 3 + c];
          if(vi[c] >= p.vertexCount)
          {
            h->err = "b200pt_set_scene: index beyond the primitive's vertex count";
            return B200PT_E_INVALID;
          }
          memcpy(&f[c * 4], &p.positions[vi[c] * 3], 12);                 // v[0..2].xyz
          if(p.normals)
            memcpy(&f[12 + c * 4], &p.normals[vi[c] * 3], 12);            // v[3..5].xyz
          if(p.colors)
            memcpy(&f[7 + c * 4], &p.colors[vi[c]], 4);                   // v[1].w, v[2].w, v[3].w
          if(p.tangents)
            memcpy(&f[36 + c * 4], &p.tangents[vi[c] * 4], 16);           // v[9..11]
        }
        if(p.texCoords[0])
        {
          f[19] = p.texCoords[0][vi[0] * 2];                               // v[4].w
          f[23] = p.texCoords[0][vi[0] * 2 + 1];                           // v[5].w
          memcpy(&f[24], &p.texCoords[0][vi[1] * 2], 8);                   // v[6].xy
          memcpy(&f[26], &p.texCoords[0][vi[2] * 2], 8);                   // v[6].zw
        }
        if(p.texCoords[1])
        {
          memcpy(&f[28], &p.texCoords[1][vi[0] * 2], 8);                   // v[7].xy
          memcpy(&f[30], &p.texCoords[1][vi[1] * 2], 8);                   // v[7].zw
          memcpy(&f[32], &p.texCoords[1][vi[2] * 2], 8);                   // v[8].xy
        }
      }
    }
    std::vector<uint32_t> idxOfSlot(bvh.numTris, 0u);
    for(uint32_t k = 0; k < bvh.numTris; k++)
    {
      uint32_t gid;
      memcpy(&gid, &bvh.tris[(size_t)k * 12 + 11], 4);
      idxOfSlot[k] = recBase[s->renderNodes[flat[gid].rnode].renderPrimID] + flat[gid].prim;
    }
    ShadeRec* dRecs;
    uint32_t* dIdx;
    if((rc = upload(h, h->sceneAllocs, recs.data(), recs.size(), &dRecs)))
      return rc;
    if((rc = upload(h, h->sceneAllocs, idxOfSlot.data(), idxOfSlot.size(), &dIdx)))
      return rc;
    S.shadeRecs = dRecs;
    S.shadeIdx = dIdx;
    h->dShadeRecsW = dRecs;
    for(uint32_t i = 0; i < s->numRenderPrimitives; i++)
      h->primHost[i].recBase = recBase[i];
    S.numMaterials = (int)s->numMaterials;
  }

  // ---- alpha-triangle records (device_scene.cuh: AlphaRec), one per non-opaque triangle in bvhA's leaf order ----
  S.alphaRecs = nullptr;
  S.alphaIdx = nullptr;
  S.alphaBaseS = 0;
  if(anyNonOpaque)
  {
    const uint32_t        nA = bvhA.numTris;
    std::vector<AlphaRec> recs(nA);
    std::vector<uint32_t> recOfGid(flat.size(), 0xFFFFFFFFu);
    for(uint32_t k = 0; k < nA; k++)
    {
      uint32_t gid;
      memcpy(&gid, &bvhA.tris[(size_t)k * 12 + 11], 4);
      recOfGid[gid] = k;
      const FlatTri&                 T = flat[gid];
      const b200pt_render_node&      node = s->renderNodes[T.rnode];
      const b200pt_render_primitive& p = s->renderPrimitives[node.renderPrimID];
      const b200pt_shade_material&   m = s->materials[(uint32_t)std::max(0, node.materialID)];
      AlphaRec                       r{};
      r.modeFlags = (uint32_t)m.alphaMode & 3u;
      r.cutoff = m.alphaCutoff;
      r.transmission = m.transmissionFactor;
      const bool     specGloss = m.pbrModel == 1;
      const uint16_t slot = specGloss ? m.pbrDiffuseTexture : m.pbrBaseColorTexture;
      r.factor = specGloss ? m.pbrDiffuseFactor[3] : m.pbrBaseColorFactor[3];
      const uint32_t i0 = p.indices[T.prim * 3], i1 = p.indices[T.prim * 3 + 1], i2 = p.indices[T.prim * 3 + 2];
      if(slot > 0)
      {
        const b200pt_texture_info& ti = s->textureInfos[slot];
        const float*               uv = ti.texCoord ? p.texCoords[1] : p.texCoords[0];
        if(uv)
        {
          const uint32_t vi[3] = {i0, i1, i2};
          for(int c = 0; c < 3; c++)
          {
            r.uv[c * 2] = uv[vi[c] * 2];
            r.uv[c * 2 + 1] = uv[vi[c] * 2 + 1];
          }
        }
        if(ti.index >= 0 && (uint32_t)ti.index < s->numTextures)
        {
          r.lv0 = texLevel0[ti.index];
          r.w0 = devTex[ti.index].w0;
          r.h0 = devTex[ti.index].h0;
          r.wrap = ((uint32_t)devTex[ti.index].wrapS & 0xffffu) | ((uint32_t)devTex[ti.index].wrapT << 16);
          if(devTex[ti.index].magLinear)
            r.modeFlags |= 4u;
        }
      }
      if(p.colors)
      {
        r.modeFlags |= 8u;
        r.colA = (p.colors[i0] >> 24) | ((p.colors[i1] >> 24) << 8) | ((p.colors[i2] >> 24) << 16);
      }
      recs[k] = r;
    }
    std::vector<uint32_t> idxOfSlot(bvh.numTris, 0xFFFFFFFFu);
    for(uint32_t k = 0; k < bvh.numTris; k++)
    {
      uint32_t gid;
      memcpy(&gid, &bvh.tris[(size_t)k * 12 + 11], 4);
      idxOfSlot[k] = recOfGid[gid];
    }
    AlphaRec* dRecs;
    uint32_t* dIdx;
    if((rc = upload(h, h->sceneAllocs, recs.data(), recs.size(), &dRecs)))
      return rc;
    if((rc = upload(h, h->sceneAllocs, idxOfSlot.data(), idxOfSlot.size(), &dIdx)))
      return rc;
    S.alphaRecs = dRecs;
    S.alphaIdx = dIdx;
    S.alphaBaseS = bvhO.numTris;
  }
  // ---- opacity micromaps (omm.cuh): one reference word per triangle slot of the merged tree and of the shadow rays' arrays ----
  h->ommTriangles = 0;
  if(anyNonOpaque && !h->primOmms.empty())
  {
    std::vector<uint8_t>  data;
    std::vector<uint32_t> dataBase(h->omms.size());
    for(size_t m = 0; m < h->omms.size(); m++)
    {
      dataBase[m] = (uint32_t)data.size();
      data.insert(data.end(), h->omms[m].data.begin(), h->omms[m].data.end());
    }
    data.resize(data.size() + 4, 0);  // (never read: keeps the allocation non-empty)
    std::vector<int> ommOfPrim(s->numRenderPrimitives, -1);
    for(size_t k = 0; k < h->primOmms.size(); k++)
    {
      const auto& po = h->primOmms[k];
      if(po.prim >= s->numRenderPrimitives)
      {
        h->err = "b200pt_set_scene: opacity micromap linked to a render primitive out of range";
        return B200PT_E_INVALID;
      }
      const uint32_t nTri = s->renderPrimitives[po.prim].triangleCount;
      if(po.hasIdx ? po.idx.size() < nTri : (uint64_t)po.base + nTri > h->omms[po.micromap].tris.size())
      {
        h->err = "b200pt_set_scene: opacity micromap does not cover its primitive's triangles";
        return B200PT_E_INVALID;
      }
      ommOfPrim[po.prim] = (int)k;
    }
    uint32_t linked = 0;
    auto     refOf = [&](uint32_t w0, uint32_t primTri) -> uint32_t {
      const uint32_t unknown = pt::kOmmNoLookup | (uint32_t)pt::OMM_UNKNOWN;
      if((w0 >> 28) & TRI_OPAQUE)
        return unknown;  // FORCE_OPAQUE instance: the walk never asks
      const int k = ommOfPrim[(uint32_t)s->renderNodes[w0 & 0x0fffffffu].renderPrimID];
      if(k < 0)
        return unknown;
      const auto& po = h->primOmms[(size_t)k];
      const int32_t idx = po.hasIdx ? po.idx[primTri] : (int32_t)primTri;
      linked++;
      if(idx == B200PT_OMM_INDEX_FULLY_TRANSPARENT)
        return pt::kOmmNoLookup | (uint32_t)pt::OMM_TRANSPARENT;
      if(idx == B200PT_OMM_INDEX_FULLY_OPAQUE)
        return pt::kOmmNoLookup | (uint32_t)pt::OMM_OPAQUE;
      if(idx < 0)
        return unknown;
      const b200pt_micromap_triangle& T = h->omms[po.micromap].tris[(size_t)idx + po.base];
      return ((uint32_t)T.subdivisionLevel << 28) | (T.format == B200PT_OMM_FORMAT_4_STATE ? (1u << 27) : 0u) | (dataBase[po.micromap] + T.dataOffset);
    };
    std::vector<uint32_t> ref(bvh.numTris), refS((size_t)bvhO.numTris + bvhA.numTris, pt::kOmmNoLookup | (uint32_t)pt::OMM_UNKNOWN);
    for(uint32_t k = 0; k < bvh.numTris; k++)
      ref[k] = refOf(bvh.triMeta[(size_t)k * 2], bvh.triMeta[(size_t)k * 2 + 1]);
    h->ommTriangles = linked;
    for(uint32_t k = 0; k < bvhA.numTris; k++)
      refS[(size_t)bvhO.numTris + k] = refOf(bvhA.triMeta[(size_t)k * 2], bvhA.triMeta[(size_t)k * 2 + 1]);
    uint8_t*  dData;
    uint32_t *dRef, *dRefS;
    if((rc = upload(h, h->sceneAllocs, data.data(), data.size(), &dData)))
      return rc;
    if((rc = upload(h, h->sceneAllocs, ref.data(), ref.size(), &dRef)))
      return rc;
    if((rc = upload(h, h->sceneAllocs, refS.data(), refS.size(), &dRefS)))
      return rc;
    S.bvh.ommRef = dRef;
    S.bvh.ommData = dData;
    S.bvhA.ommRef = dRefS;
    S.bvhA.ommData = dData;
  }
  h->nodeBytes = bvh.nodes.size() * sizeof(float) + splitNodeBytes;
  h->triBytes = bvh.tris.size() * sizeof(float) + splitTriBytes;
  h->numNodes = bvh.numNodes + (anyNonOpaque ? bvhO.numNodes + bvhA.numNodes : 0u);
  h->numTris = bvh.numTris;
  CK(cudaStreamSynchronize(h->stream));
  h->haveScene = true;
  // Persisting-L2 window over the trees on every stream that runs walks (cudaAccessPolicyWindow: lines of the window are kept, the
  // path-state traffic around them is what gets evicted).  hitRatio shrinks when the trees are larger than the carve-out.
  if(h->treeBytes)
  {
    int maxPersist = 0, maxWindow = 0;
    cudaDeviceGetAttribute(&maxPersist, cudaDevAttrMaxPersistingL2CacheSize, h->device);
    cudaDeviceGetAttribute(&maxWindow, cudaDevAttrMaxAccessPolicyWindowSize, h->device);
    if(maxPersist > 0 && maxWindow > 0)
    {
      const size_t carve = std::min<size_t>((size_t)maxPersist, std::max<size_t>(h->treeBytes, (size_t)1 << 20));
      cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
      cudaStreamAttrValue attr{};
      attr.accessPolicyWindow.base_ptr = const_cast<void*>(h->treeBase);
      attr.accessPolicyWindow.num_bytes = std::min<size_t>(h->treeBytes, (size_t)maxWindow);
      attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)carve / (double)attr.accessPolicyWindow.num_bytes);
      attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
      cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &attr);
      for(int l = 0; l < b200pt::kMaxLanes; l++)
        if(h->lanes[l].stream)
          cudaStreamSetAttribute(h->lanes[l].stream, cudaStreamAttributeAccessPolicyWindow, &attr);
      cudaGetLastError();  // (a refused window is not an error: the walks run without it)
    }
  }
  return B200PT_OK;
}

int b200pt_bvh_info(b200pt_t* h, uint64_t* node_bytes, uint64_t* tri_bytes, uint32_t* num_nodes, uint32_t* num_tris)
{
  if(!h || !h->haveScene)
    return B200PT_E_INVALID;
  if(node_bytes)
    *node_bytes = h->nodeBytes;
  if(tri_bytes)
    *tri_bytes = h->triBytes;
  if(num_nodes)
    *num_nodes = h->numNodes;
  if(num_tris)
    *num_tris = h->numTris;
  return B200PT_OK;
}

int b200pt_set_opacity_micromaps(b200pt_t* h, const b200pt_micromap* micromaps, uint32_t num_micromaps, const b200pt_primitive_omm* prims, uint32_t num_prims)
{
  if(!h || (num_micromaps && !micromaps) || (num_prims && !prims))
    return B200PT_E_INVALID;
  std::vector<b200pt_t::OmmHost>     omms(num_prims ? num_micromaps : 0u);
  std::vector<b200pt_t::PrimOmmHost> po(num_prims);
  uint64_t                           total = 0;
  for(size_t m = 0; m < omms.size(); m++)
  {
    const b200pt_micromap& M = micromaps[m];
    if((M.dataSize && !M.data) || (M.numTriangles && !M.triangles))
    {
      h->err = "b200pt_set_opacity_micromaps: micromap with a null array";
      return B200PT_E_INVALID;
    }
    for(uint32_t t = 0; t < M.numTriangles; t++)
    {
      const b200pt_micromap_triangle& T = M.triangles[t];
      if((T.format != B200PT_OMM_FORMAT_2_STATE && T.format != B200PT_OMM_FORMAT_4_STATE) || T.subdivisionLevel > B200PT_OMM_MAX_LEVEL)
      {
        h->err = "b200pt_set_opacity_micromaps: micromap triangle with an unknown format or a subdivision level above 12";
        return B200PT_E_INVALID;
      }
      const uint64_t bits = (1ull << (2 * T.subdivisionLevel)) * (T.format == B200PT_OMM_FORMAT_4_STATE ? 2u : 1u);
      if((uint64_t)T.dataOffset + (bits + 7) / 8 > M.dataSize)
      {
        h->err = "b200pt_set_opacity_micromaps: micromap triangle data beyond dataSize";
        return B200PT_E_INVALID;
      }
    }
    omms[m].data.assign(M.data, M.data + M.dataSize);
    omms[m].tris.assign(M.triangles, M.triangles + M.numTriangles);
    total += M.dataSize;
  }
  if(total >= (1ull << 27))
  {
    h->err = "b200pt_set_opacity_micromaps: more than 128 MiB of micromap data";
    return B200PT_E_UNSUPPORTED;
  }
  for(uint32_t i = 0; i < num_prims; i++)
  {
    const b200pt_primitive_omm& P = prims[i];
    if(P.micromap >= num_micromaps || (P.numIndices && !P.indices))
    {
      h->err = "b200pt_set_opacity_micromaps: primitive linkage references a micromap out of range";
      return B200PT_E_INVALID;
    }
    po[i].prim = P.renderPrimID;
    po[i].micromap = P.micromap;
    po[i].base = P.baseTriangle;
    po[i].hasIdx = P.indices != nullptr;
    if(P.indices)
      po[i].idx.assign(P.indices, P.indices + P.numIndices);
    for(int32_t v : po[i].idx)
      if(v < B200PT_OMM_INDEX_FULLY_UNKNOWN_OPAQUE || (v >= 0 && (uint64_t)v + P.baseTriangle >= micromaps[P.micromap].numTriangles))
      {
        h->err = "b200pt_set_opacity_micromaps: micromap index out of range";
        return B200PT_E_INVALID;
      }
  }
  h->omms.swap(omms);
  h->primOmms.swap(po);
  return B200PT_OK;
}

int b200pt_set_bvh_builder(b200pt_t* h, int kind)
{
  if(!h || (kind != 0 && kind != 1))
    return B200PT_E_INVALID;
  h->bvhBuilder = kind;
  return B200PT_OK;
}

int b200pt_bvh_build_ms(b200pt_t* h, double* ms)
{
  if(!h || !ms || !h->haveScene)
    return B200PT_E_INVALID;
  *ms = h->bvhBuildMs;
  return B200PT_OK;
}

// triangle records recomputed from the primitives' current vertices and the nodes' current transforms, then every tree
// refitted bottom-up (refit.cuh); synchronous
static int refitTrees(b200pt_t* h)
{
  cudaStream_t st = h->stream;
  for(int t = 0; t < 3; t++)
  {
    b200pt::TreeDev& T = h->tree[t];
    if(!T.nodes)
      continue;
    if(T.numTriSlots)
    {
      k_refit_tris<<<gridFor(h, 4), 256, 0, st>>>(T.tris, T.meta, T.numTriSlots, h->dNodesW, h->dPrimsW);
      h->kernelLaunches++;
    }
  }
  for(int t = 0; t < 3; t++)
  {
    b200pt::TreeDev& T = h->tree[t];
    if(!T.nodes)
      continue;
    for(size_t l = T.levels.size(); l-- > 0;)
    {
      const uint32_t count = T.levels[l].second;
      k_refit_level<<<(count + 127) / 128, 128, 0, st>>>(T.nodes, T.tris, T.nodeBox, T.levels[l].first, count);
      h->kernelLaunches++;
    }
  }
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st));
  return B200PT_OK;
}

int b200pt_update_transforms(b200pt_t* h, const b200pt_render_node* nodes, uint32_t num_nodes)
{
  if(!h || !h->haveScene || !nodes || num_nodes != h->numSceneNodes)
  {
    if(h)
      h->err = "b200pt_update_transforms: needs the scene's render-node count (materials / primitives of the nodes must not change)";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  cudaStream_t st = h->stream;
  CK(cudaMemcpyAsync(h->dNodesW, nodes, (size_t)num_nodes * sizeof(b200pt_render_node), cudaMemcpyHostToDevice, st));
  return refitTrees(h);
}

int b200pt_set_node_hierarchy(b200pt_t* h, const b200pt_node_hierarchy* g)
{
  if(!h || !h->haveScene || !g || g->numNodes == 0 || g->numLevels == 0 || !g->parentIndices || !g->topoNodeOrder || !g->levelOffsets || !g->mappings)
  {
    if(h)
      h->err = "b200pt_set_node_hierarchy: needs a scene and a complete hierarchy description";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  freeHierarchy(h);
  auto fail = [&](const char* msg) {
    freeHierarchy(h);
    h->err = msg;
    return B200PT_E_INVALID;
  };
  // every node exactly once, parents in earlier levels, offsets monotone and complete
  if(g->levelOffsets[0] != 0 || g->levelOffsets[g->numLevels] != g->numNodes)
    return fail("b200pt_set_node_hierarchy: levelOffsets must run from 0 to numNodes");
  std::vector<int> levelOf(g->numNodes, -1);
  for(uint32_t l = 0; l < g->numLevels; l++)
  {
    if(g->levelOffsets[l + 1] < g->levelOffsets[l] || g->levelOffsets[l + 1] > g->numNodes)
      return fail("b200pt_set_node_hierarchy: levelOffsets must be monotone");
    for(uint32_t k = g->levelOffsets[l]; k < g->levelOffsets[l + 1]; k++)
    {
      const int n = g->topoNodeOrder[k];
      if(n < 0 || (uint32_t)n >= g->numNodes || levelOf[n] != -1)
        return fail("b200pt_set_node_hierarchy: topoNodeOrder must list every node once");
      levelOf[n] = (int)l;
    }
  }
  for(uint32_t n = 0; n < g->numNodes; n++)
  {
    const int p = g->parentIndices[n];
    if(p >= (int)g->numNodes || (p >= 0 && levelOf[p] >= levelOf[n]))
      return fail("b200pt_set_node_hierarchy: a parent must sit in an earlier level than its child");
  }
  for(uint32_t i = 0; i < h->numSceneNodes; i++)
  {
    const b200pt_render_node_mapping& m = g->mappings[i];
    if(m.nodeID < 0 || (uint32_t)m.nodeID >= g->numNodes || m.renderPrimID < 0 || (size_t)m.renderPrimID >= h->primHost.size() || m.materialID >= h->S.numMaterials)
      return fail("b200pt_set_node_hierarchy: render-node mapping out of range");
  }
  int rc;
  if((rc = upload(h, h->graphAllocs, g->parentIndices, g->numNodes, &h->dParents)))
    return rc;
  if((rc = upload(h, h->graphAllocs, g->topoNodeOrder, g->numNodes, &h->dTopo)))
    return rc;
  static_assert(sizeof(RenderNodeMapping) == sizeof(b200pt_render_node_mapping), "mapping layout");
  if((rc = upload(h, h->graphAllocs, reinterpret_cast<const RenderNodeMapping*>(g->mappings), h->numSceneNodes, &h->dMappings)))
    return rc;
  if(g->instLocalMatrices && (rc = upload(h, h->graphAllocs, g->instLocalMatrices, (size_t)h->numSceneNodes * 16, &h->dInstLocal)))
    return rc;
  CK(cudaMalloc((void**)&h->dLocalMats, (size_t)g->numNodes * 16 * sizeof(float)));
  h->graphAllocs.push_back(h->dLocalMats);
  CK(cudaMalloc((void**)&h->dWorldMats, (size_t)g->numNodes * 16 * sizeof(float)));
  h->graphAllocs.push_back(h->dWorldMats);
  h->levelOffsets.assign(g->levelOffsets, g->levelOffsets + g->numLevels + 1);
  h->numGraphNodes = g->numNodes;
  CK(cudaStreamSynchronize(h->stream));
  return B200PT_OK;
}

int b200pt_update_node_matrices(b200pt_t* h, const float* local_matrices)
{
  if(!h || !h->haveScene || h->numGraphNodes == 0 || !local_matrices)
  {
    if(h)
      h->err = "b200pt_update_node_matrices: needs b200pt_set_node_hierarchy and the nodes' local matrices";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  cudaStream_t st = h->stream;
  CK(cudaMemcpyAsync(h->dLocalMats, local_matrices, (size_t)h->numGraphNodes * 16 * sizeof(float), cudaMemcpyHostToDevice, st));
  for(size_t l = 0; l + 1 < h->levelOffsets.size(); l++)
  {
    const uint32_t count = h->levelOffsets[l + 1] - h->levelOffsets[l];
    if(!count)
      continue;
    k_propagate_level<<<(count + 255) / 256, 256, 0, st>>>(h->dLocalMats, h->dWorldMats, h->dParents, h->dTopo, h->levelOffsets[l], count);
    h->kernelLaunches++;
  }
  if(h->numSceneNodes)
  {
    k_update_render_nodes<<<(h->numSceneNodes + 255) / 256, 256, 0, st>>>(h->dWorldMats, h->dMappings, h->dInstLocal, h->dNodesW, h->numSceneNodes);
    h->kernelLaunches++;
  }
  CK(cudaGetLastError());
  return refitTrees(h);
}

int b200pt_set_animation(b200pt_t* h, const b200pt_morph_task* morphs, uint32_t num_morphs, const b200pt_skin_task* skins, uint32_t num_skins)
{
  if(!h || !h->haveScene || (num_morphs && !morphs) || (num_skins && !skins))
  {
    if(h)
      h->err = "b200pt_set_animation: needs a scene (b200pt_set_scene first) and task arrays";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  freeAnimation(h);
  auto fail = [&](const char* msg) {
    freeAnimation(h);
    h->err = msg;
    return B200PT_E_INVALID;
  };
  int rc;
  for(uint32_t i = 0; i < num_morphs; i++)
  {
    const b200pt_morph_task& m = morphs[i];
    if(m.renderPrimID >= h->primHost.size())
      return fail("b200pt_set_animation: morph task for a render primitive out of range");
    const b200pt::PrimHost& P = h->primHost[m.renderPrimID];
    if(m.vertexCount != P.vertexCount || !m.basePositions || (m.numTargets && !m.positionDeltas))
      return fail("b200pt_set_animation: morph task needs base positions, position deltas and the primitive's vertex count");
    MorphTaskDev T{};
    T.vertexCount = m.vertexCount;
    T.numTargets = m.numTargets;
    const size_t nv = m.vertexCount, nd = (size_t)m.numTargets * m.vertexCount * 3;
    float*       d;
    if((rc = upload(h, h->animAllocs, m.basePositions, nv * 3, &d)))
      return rc;
    T.basePos = d;
    if(m.baseNormals && P.d.nrm)
    {
      if((rc = upload(h, h->animAllocs, m.baseNormals, nv * 3, &d)))
        return rc;
      T.baseNrm = d;
    }
    if(m.baseTangents && P.d.tan)
    {
      if((rc = upload(h, h->animAllocs, m.baseTangents, nv * 4, &d)))
        return rc;
      T.baseTan = d;
    }
    if((rc = upload(h, h->animAllocs, m.positionDeltas, nd, &d)))
      return rc;
    T.dPos = d;
    if(m.normalDeltas && T.baseNrm)
    {
      if((rc = upload(h, h->animAllocs, m.normalDeltas, nd, &d)))
        return rc;
      T.dNrm = d;
    }
    if(m.tangentDeltas && T.baseTan)
    {
      if((rc = upload(h, h->animAllocs, m.tangentDeltas, nd, &d)))
        return rc;
      T.dTan = d;
    }
    T.outPos = const_cast<float*>(P.d.pos);
    T.outNrm = const_cast<float*>(P.d.nrm);
    T.outTan = const_cast<float*>(P.d.tan);
    h->numMorphWeights += m.numTargets;
    h->morphTasks.push_back(T);
    h->morphPrim.push_back(m.renderPrimID);
  }
  for(uint32_t i = 0; i < num_skins; i++)
  {
    const b200pt_skin_task& k = skins[i];
    if(k.renderPrimID >= h->primHost.size())
      return fail("b200pt_set_animation: skin task for a render primitive out of range");
    const b200pt::PrimHost& P = h->primHost[k.renderPrimID];
    if(k.vertexCount != P.vertexCount || !k.basePositions || !k.weights || !k.joints || k.numJoints == 0)
      return fail("b200pt_set_animation: skin task needs base positions, weights, joints and the primitive's vertex count");
    SkinTaskDev  T{};
    const size_t nv = k.vertexCount;
    T.vertexCount = k.vertexCount;
    T.numJoints = k.numJoints;
    float* d;
    int*   di;
    if((rc = upload(h, h->animAllocs, k.basePositions, nv * 3, &d)))
      return rc;
    T.basePos = d;
    if(k.baseNormals && P.d.nrm)
    {
      if((rc = upload(h, h->animAllocs, k.baseNormals, nv * 3, &d)))
        return rc;
      T.baseNrm = d;
    }
    if(k.baseTangents && P.d.tan)
    {
      if((rc = upload(h, h->animAllocs, k.baseTangents, nv * 4, &d)))
        return rc;
      T.baseTan = d;
    }
    if((rc = upload(h, h->animAllocs, k.weights, nv * 4, &d)))
      return rc;
    T.weights = d;
    if((rc = upload(h, h->animAllocs, k.joints, nv * 4, &di)))
      return rc;
    T.joints = di;
    T.outPos = const_cast<float*>(P.d.pos);
    T.outNrm = const_cast<float*>(P.d.nrm);
    T.outTan = const_cast<float*>(P.d.tan);
    h->numJoints += k.numJoints;
    h->skinTasks.push_back(T);
    h->skinPrim.push_back(k.renderPrimID);
  }
  // the per-frame buffers, sized once (createAnimationResources: totalJointMatBytes / totalNormalMatBytes / morph weights)
  CK(cudaMalloc((void**)&h->dMorphWeights, std::max<size_t>(h->numMorphWeights, 1) * sizeof(float)));
  h->animAllocs.push_back(h->dMorphWeights);
  CK(cudaMalloc((void**)&h->dJointMats, std::max<size_t>(h->numJoints, 1) * 16 * sizeof(float)));
  h->animAllocs.push_back(h->dJointMats);
  CK(cudaMalloc((void**)&h->dNormalMats, std::max<size_t>(h->numJoints, 1) * 9 * sizeof(float)));
  h->animAllocs.push_back(h->dNormalMats);
  size_t wOfs = 0, jOfs = 0;
  for(auto& T : h->morphTasks)
  {
    T.weights = h->dMorphWeights + wOfs;
    wOfs += T.numTargets;
  }
  for(auto& T : h->skinTasks)
  {
    T.jointMatrices = h->dJointMats + jOfs * 16;
    T.normalMatrices = h->dNormalMats + jOfs * 9;
    jOfs += T.numJoints;
  }
  CK(cudaStreamSynchronize(h->stream));
  return B200PT_OK;
}

int b200pt_animate(b200pt_t* h, const float* morph_weights, const float* joint_matrices, const float* normal_matrices)
{
  if(!h || !h->haveScene || (h->morphTasks.empty() && h->skinTasks.empty()) || (h->numMorphWeights && !morph_weights)
     || (h->numJoints && (!joint_matrices || !normal_matrices)))
  {
    if(h)
      h->err = "b200pt_animate: needs b200pt_set_animation and the per-frame weights / joint matrices / normal matrices of its tasks";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  cudaStream_t st = h->stream;
  // Phase 1 (gltf_scene_animation_vk.cpp:430-494): one upload of all per-frame data
  if(h->numMorphWeights)
    CK(cudaMemcpyAsync(h->dMorphWeights, morph_weights, h->numMorphWeights * sizeof(float), cudaMemcpyHostToDevice, st));
  if(h->numJoints)
  {
    CK(cudaMemcpyAsync(h->dJointMats, joint_matrices, h->numJoints * 16 * sizeof(float), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->dNormalMats, normal_matrices, h->numJoints * 9 * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  // Phase 2 (:497-533): morph
  std::vector<uint8_t> touched(h->primHost.size(), 0), morphed(h->primHost.size(), 0);
  for(size_t i = 0; i < h->morphTasks.size(); i++)
  {
    const MorphTaskDev& T = h->morphTasks[i];
    if(T.numTargets == 0)
      continue;  // (:508) nothing to blend: the vertex buffers keep what they hold
    k_morph<<<(T.vertexCount + 255) / 256, 256, 0, st>>>(T);
    h->kernelLaunches++;
    touched[h->morphPrim[i]] = morphed[h->morphPrim[i]] = 1;
  }
  // Phase 3 (:536-582): skin; a primitive morphed above is skinned from its own (morphed) arrays
  for(size_t i = 0; i < h->skinTasks.size(); i++)
  {
    SkinTaskDev T = h->skinTasks[i];
    if(morphed[h->skinPrim[i]])
    {
      const DevPrim& P = h->primHost[h->skinPrim[i]].d;
      T.basePos = P.pos;
      T.baseNrm = P.nrm ? P.nrm : T.baseNrm;
      T.baseTan = P.tan ? P.tan : T.baseTan;
    }
    k_skin<<<(T.vertexCount + 255) / 256, 256, 0, st>>>(T);
    h->kernelLaunches++;
    touched[h->skinPrim[i]] = 1;
  }
  // the per-triangle shade records of the touched primitives follow their vertex arrays
  for(size_t p = 0; p < touched.size(); p++)
    if(touched[p] && h->primHost[p].triCount)
    {
      const b200pt::PrimHost& P = h->primHost[p];
      k_regather_shade<<<(P.triCount + 255) / 256, 256, 0, st>>>(h->dShadeRecsW + P.recBase, P.d, P.triCount);
      h->kernelLaunches++;
    }
  CK(cudaGetLastError());
  // the BLAS update the reference records after the compute barrier (:586-590): triangle records + bottom-up refit
  return refitTrees(h);
}

int b200pt_set_environment(b200pt_t* h, const float* rgb, int w, int hh, float* integral_out)
{
  if(!h || !rgb || w <= 0 || hh <= 0)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  const size_t n = (size_t)w * hh;
  // importance = texel solid angle * max(r,g,b); Vose alias table; pdf stored in alpha
  // (nvvk::HdrIbl, external to the reference tree; call site src/renderer.cpp:1994-1996)
  std::vector<float>  rgba(n * 4), importance(n), q(n);
  std::vector<uint32_t> alias(n);
  const float         stepPhi = kTwoPi / (float)w, stepTheta = kPi / (float)hh;
  for(int y = 0; y < hh; y++)
  {
    const float theta0 = (float)y * stepTheta, theta1 = (float)(y + 1) * stepTheta;
    const float area = (cosf(theta0) - cosf(theta1)) * stepPhi;
    for(int x = 0; x < w; x++)
    {
      const size_t i = (size_t)y * w + x;
      const float  r = rgb[i * 3], g = rgb[i * 3 + 1], b = rgb[i * 3 + 2];
      rgba[i * 4] = r;
      rgba[i * 4 + 1] = g;
      rgba[i * 4 + 2] = b;
      importance[i] = area * std::max(r, std::max(g, b));
    }
  }
  float sum = 0.f;
  for(float d : importance)
    sum += d;
  const float average = sum / (float)n;
  for(size_t i = 0; i < n; i++)
  {
    q[i] = importance[i] / average;
    alias[i] = (uint32_t)i;
  }
  {
    std::vector<uint32_t> part(n);
    uint32_t              s = 0u, large = (uint32_t)n;
    for(uint32_t i = 0; i < (uint32_t)n; ++i)
    {
      if(q[i] < 1.f)
        part[s++] = i;
      else
        part[--large] = i;
    }
    for(s = 0; s < large && large < (uint32_t)n; ++s)
    {
      const uint32_t j = part[s], k = part[large];
      alias[j] = k;
      const float diff = 1.f - q[j];
      q[k] -= diff;
      if(q[k] < 1.0f)
        large++;
    }
  }
  const float inv = 1.0f / sum;
  for(size_t i = 0; i < n; i++)
    rgba[i * 4 + 3] = std::max(rgba[i * 4], std::max(rgba[i * 4 + 1], rgba[i * 4 + 2])) * inv;
  std::vector<uint32_t> accel(n * 2);
  for(size_t i = 0; i < n; i++)
  {
    accel[i * 2] = alias[i];
    memcpy(&accel[i * 2 + 1], &q[i], 4);
  }
  if(h->dEnv)
    cudaFree(h->dEnv);
  if(h->dEnvAccel)
    cudaFree(h->dEnvAccel);
  h->dEnv = nullptr;
  h->dEnvAccel = nullptr;
  CK(cudaMalloc((void**)&h->dEnv, n * sizeof(float4)));
  CK(cudaMalloc((void**)&h->dEnvAccel, n * sizeof(uint2)));
  CK(cudaMemcpy(h->dEnv, rgba.data(), n * sizeof(float4), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->dEnvAccel, accel.data(), n * sizeof(uint2), cudaMemcpyHostToDevice));
  h->S.envRgba = h->dEnv;
  h->S.envAccel = h->dEnvAccel;
  h->S.envW = w;
  h->S.envH = hh;
  h->haveEnv = true;
  if(integral_out)
    *integral_out = sum;
  return B200PT_OK;
}

int b200pt_resize(b200pt_t* h, int width, int height, int tile_y0, int tile_rows)
{
  if(!h || width <= 0 || height <= 0 || tile_y0 < 0 || tile_rows <= 0 || tile_y0 + tile_rows > height)
  {
    if(h)
      h->err = "b200pt_resize: invalid extent / tile";
    return B200PT_E_INVALID;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  freePool(h);
  const size_t n = (size_t)width * tile_rows;          // pixels of the tile: image-sized buffers
  const size_t nPool = n * (size_t)std::max(h->batch, 1);  // path slots per lane
  // nothing of the handle's geometry is committed before every allocation has succeeded: a failed resize leaves
  // numPaths == 0 and null pointers, so later calls fail their guards instead of touching freed memory
  auto fail = [&](int rc) {
    freePool(h);
    return rc;
  };
  for(int l = 0; l < h->numLanes; l++)
  {
    b200pt::Lane& L = h->lanes[l];
    const int     rc = allocPathState(h, h->poolAllocs, nPool, L.P);
    if(rc)
      return fail(rc);
    for(int k = 0; k < 6; k++)
    {
      if(cudaMalloc((void**)&L.dQ[k], nPool * sizeof(uint32_t)) != cudaSuccess)
      {
        cudaGetLastError();
        L.dQ[k] = nullptr;
        h->err = "path pool: out of device memory";
        return fail(B200PT_E_NOMEM);
      }
      h->poolAllocs.push_back(L.dQ[k]);
    }
  }
  if(cudaMalloc((void**)&h->dAccumOwned, n * 16) != cudaSuccess)
  {
    cudaGetLastError();
    h->err = "accumulation image: out of device memory";
    return fail(B200PT_E_NOMEM);
  }
  h->poolAllocs.push_back(h->dAccumOwned);
  if(cudaMalloc((void**)&h->dSelect, n * 4) != cudaSuccess)
  {
    cudaGetLastError();
    h->dSelect = nullptr;
    h->err = "selection image: out of device memory";
    return fail(B200PT_E_NOMEM);
  }
  h->poolAllocs.push_back(h->dSelect);
  if(cudaMalloc((void**)&h->dNdcDepth, n * 4) != cudaSuccess)
  {
    cudaGetLastError();
    h->dNdcDepth = nullptr;
    h->err = "depth image: out of device memory";
    return fail(B200PT_E_NOMEM);
  }
  h->poolAllocs.push_back(h->dNdcDepth);
  if(h->guides)
  {
    if(cudaMalloc((void**)&h->dGuide, n * 16) != cudaSuccess)
    {
      cudaGetLastError();
      h->dGuide = nullptr;
      h->err = "guide image: out of device memory";
      return fail(B200PT_E_NOMEM);
    }
    h->poolAllocs.push_back(h->dGuide);
    if(cudaMemsetAsync(h->dGuide, 0, n * 16, h->stream) != cudaSuccess)
      return fail(B200PT_E_CUDA);
  }
  if(cudaMalloc((void**)&h->dTonemapped, n * 4) != cudaSuccess)
  {
    cudaGetLastError();
    h->dTonemapped = nullptr;
    h->err = "tonemapped image: out of device memory";
    return fail(B200PT_E_NOMEM);
  }
  h->poolAllocs.push_back(h->dTonemapped);
  if(cudaMemsetAsync(h->dSelect, 0, n * 4, h->stream) != cudaSuccess || cudaMemsetAsync(h->dNdcDepth, 0, n * 4, h->stream) != cudaSuccess
     || cudaMemsetAsync(h->dAccumOwned, 0, n * 16, h->stream) != cudaSuccess || cudaStreamSynchronize(h->stream) != cudaSuccess)
  {
    h->err = "b200pt_resize: clearing the accumulation image failed";
    return fail(B200PT_E_CUDA);
  }
  h->width = width;
  h->height = height;
  h->tileY0 = tile_y0;
  h->tileRows = tile_rows;
  h->bandRows = 0;
  h->bandWorld = 1;
  h->bandRank = 0;
  h->numPaths = (uint32_t)n;
  h->dAccum = h->dAccumOwned;
  return B200PT_OK;
}

int b200pt_resize_interleaved(b200pt_t* h, int width, int height, int band_rows, int world, int rank)
{
  if(!h || width <= 0 || height <= 0 || band_rows <= 0 || world <= 0 || rank < 0 || rank >= world || height % (band_rows * world) != 0)
  {
    if(h)
      h->err = "b200pt_resize_interleaved: height must be a multiple of band_rows * world, 0 <= rank < world";
    return B200PT_E_INVALID;
  }
  const int rc = b200pt_resize(h, width, height, 0, height / world);
  if(rc)
    return rc;
  h->bandRows = band_rows;
  h->bandWorld = world;
  h->bandRank = rank;
  return B200PT_OK;
}

int b200pt_set_accum_device(b200pt_t* h, float* dev, size_t num_floats)
{
  if(!h || h->numPaths == 0)
    return B200PT_E_INVALID;
  if(dev == nullptr)
  {
    h->dAccum = h->dAccumOwned;
    return B200PT_OK;
  }
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  if(num_floats < (size_t)h->numPaths * 4)
  {
    h->err = "b200pt_set_accum_device: buffer too small";
    return B200PT_E_INVALID;
  }
  h->dAccum = reinterpret_cast<float4*>(dev);
  return B200PT_OK;
}

int b200pt_get_accum_device(b200pt_t* h, float** dev, size_t* num_floats)
{
  if(!h || h->numPaths == 0)
    return B200PT_E_INVALID;
  if(dev)
    *dev = reinterpret_cast<float*>(h->dAccum);
  if(num_floats)
    *num_floats = (size_t)h->numPaths * 4;
  return B200PT_OK;
}

int b200pt_read_accum(b200pt_t* h, float* host, size_t num_floats)
{
  if(!h || h->numPaths == 0 || !host || num_floats < (size_t)h->numPaths * 4)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  CK(cudaMemcpyAsync(host, h->dAccum, (size_t)h->numPaths * 16, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return B200PT_OK;
}

// histogram (when auto-exposure is on) -> exposure factor -> operator + UNORM8 store, on the handle's stream
static int tonemapOnDevice(b200pt_t* h, const b200pt_tonemapper* tm, const float4* img, int width, int rows, int y0, int fullHeight, uchar4* out, float* exposure_used)
{
  if(tm->method < 0 || tm->method > 5 || !(tm->brightness > 0.0f))
  {
    h->err = "b200pt_tonemap: method must be 0..5 and brightness > 0";
    return B200PT_E_INVALID;
  }
  cudaStream_t   st = h->stream;
  const uint32_t n = (uint32_t)width * (uint32_t)rows;
  float*         dExposure = reinterpret_cast<float*>(h->dTmHist + kTmBins);
  if(tm->autoExposure && tm->isActive)
  {
    CK(cudaMemsetAsync(h->dTmHist, 0, kTmBins * sizeof(uint32_t), st));
    k_tm_histogram<<<gridFor(h, 8), 256, 0, st>>>(img, n, h->dTmHist);
    k_tm_exposure<<<1, 32, 0, st>>>(h->dTmHist, tm->exposure, dExposure);
    h->kernelLaunches += 2;
  }
  else
    CK(cudaMemcpyAsync(dExposure, &tm->exposure, sizeof(float), cudaMemcpyHostToDevice, st));
  k_tonemap<<<gridFor(h, 8), 256, 0, st>>>(img, out, width, rows, y0, fullHeight, *tm, dExposure);
  h->kernelLaunches++;
  CK(cudaGetLastError());
  if(exposure_used)
    CK(cudaMemcpyAsync(exposure_used, dExposure, sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return B200PT_OK;
}

int b200pt_tonemap(b200pt_t* h, const b200pt_tonemapper* tm, uint8_t* host_rgba8, size_t num_bytes, float* exposure_used)
{
  if(!h || !tm || h->numPaths == 0 || (host_rgba8 && num_bytes < (size_t)h->numPaths * 4))
    return B200PT_E_INVALID;
  if(h->bandWorld > 1)
  {
    h->err = "b200pt_tonemap: an interleaved multi-GPU tile is tonemapped after the gather (b200pt_tonemap_image on the full image)";
    return B200PT_E_UNSUPPORTED;
  }
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  const int rc = tonemapOnDevice(h, tm, h->dAccum, h->width, h->tileRows, h->tileY0, h->height, h->dTonemapped, exposure_used);
  if(rc)
    return rc;
  if(host_rgba8)
  {
    CK(cudaMemcpyAsync(host_rgba8, h->dTonemapped, (size_t)h->numPaths * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return B200PT_OK;
}

int b200pt_tonemap_image(b200pt_t* h, const b200pt_tonemapper* tm, const float* dev_rgba32f, int width, int height, uint8_t* dev_rgba8, float* exposure_used)
{
  if(!h || !tm || !dev_rgba32f || !dev_rgba8 || width <= 0 || height <= 0)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  return tonemapOnDevice(h, tm, reinterpret_cast<const float4*>(dev_rgba32f), width, height, 0, height, reinterpret_cast<uchar4*>(dev_rgba8), exposure_used);
}

int b200pt_get_tonemapped_device(b200pt_t* h, uint8_t** dev_rgba8, size_t* num_bytes)
{
  if(!h || h->numPaths == 0 || !dev_rgba8)
    return B200PT_E_INVALID;
  *dev_rgba8 = reinterpret_cast<uint8_t*>(h->dTonemapped);
  if(num_bytes)
    *num_bytes = (size_t)h->numPaths * 4;
  return B200PT_OK;
}

int b200pt_read_selection(b200pt_t* h, uint32_t* host_object_ids, float* host_ndc_depth, size_t num_pixels)
{
  if(!h || h->numPaths == 0 || num_pixels < (size_t)h->numPaths || (!host_object_ids && !host_ndc_depth))
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  if(host_object_ids)
    CK(cudaMemcpyAsync(host_object_ids, h->dSelect, (size_t)h->numPaths * 4, cudaMemcpyDeviceToHost, h->stream));
  if(host_ndc_depth)
    CK(cudaMemcpyAsync(host_ndc_depth, h->dNdcDepth, (size_t)h->numPaths * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return B200PT_OK;
}

int b200pt_get_selection_device(b200pt_t* h, uint32_t** dev_object_ids, float** dev_ndc_depth)
{
  if(!h || h->numPaths == 0)
    return B200PT_E_INVALID;
  if(dev_object_ids)
    *dev_object_ids = h->dSelect;
  if(dev_ndc_depth)
    *dev_ndc_depth = h->dNdcDepth;
  return B200PT_OK;
}

int b200pt_read_accum_async(b200pt_t* h, float* host, size_t num_floats, int slot)
{
  if(!h || h->numPaths == 0 || !host || num_floats < (size_t)h->numPaths * 4 || slot < 0 || slot >= 8)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  if(!h->readDone[slot])
    CK(cudaEventCreateWithFlags(&h->readDone[slot], cudaEventDisableTiming));
  else
    CK(cudaEventSynchronize(h->readDone[slot]));
  CK(cudaMemcpyAsync(host, h->dAccum, (size_t)h->numPaths * 16, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaEventRecord(h->readDone[slot], h->stream));
  return B200PT_OK;
}

int b200pt_wait_read(b200pt_t* h, int slot)
{
  if(!h || slot < 0 || slot >= 8)
    return B200PT_E_INVALID;
  if(h->readDone[slot])
    CK(cudaEventSynchronize(h->readDone[slot]));
  return B200PT_OK;
}

int b200pt_set_frames_in_flight(b200pt_t* h, int n)
{
  if(!h || n < 1 || n > b200pt::kMaxLanes)
    return B200PT_E_INVALID;
  if(n == h->numLanes)
    return B200PT_OK;
  h->numLanes = n;
  if(h->numPaths == 0)
    return B200PT_OK;
  float4* const user = (h->dAccum != h->dAccumOwned) ? h->dAccum : nullptr;
  int           rc;
  if(h->bandWorld > 1)
    rc = b200pt_resize_interleaved(h, h->width, h->height, h->bandRows, h->bandWorld, h->bandRank);
  else
    rc = b200pt_resize(h, h->width, h->height, h->tileY0, h->tileRows);
  if(rc == B200PT_OK && user)
    h->dAccum = user;
  return rc;
}

int b200pt_set_guide_outputs(b200pt_t* h, int enable)
{
  if(!h)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  if((enable != 0) == h->guides)
    return B200PT_OK;
  h->guides = enable != 0;
  if(h->numPaths == 0)
    return B200PT_OK;
  float4* const user = (h->dAccum != h->dAccumOwned) ? h->dAccum : nullptr;
  int           rc;
  if(h->bandWorld > 1)
    rc = b200pt_resize_interleaved(h, h->width, h->height, h->bandRows, h->bandWorld, h->bandRank);
  else
    rc = b200pt_resize(h, h->width, h->height, h->tileY0, h->tileRows);
  if(rc == B200PT_OK && user)
    h->dAccum = user;
  return rc;
}

int b200pt_read_guide(b200pt_t* h, float* host_albedo_normal, size_t num_floats)
{
  if(!h || h->numPaths == 0 || !h->dGuide || !host_albedo_normal || num_floats < (size_t)h->numPaths * 4)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  CK(cudaMemcpyAsync(host_albedo_normal, h->dGuide, (size_t)h->numPaths * 16, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return B200PT_OK;
}

int b200pt_get_guide_device(b200pt_t* h, float** dev_albedo_normal, size_t* num_floats)
{
  if(!h || h->numPaths == 0 || !h->dGuide || !dev_albedo_normal)
    return B200PT_E_INVALID;
  *dev_albedo_normal = reinterpret_cast<float*>(h->dGuide);
  if(num_floats)
    *num_floats = (size_t)h->numPaths * 4;
  return B200PT_OK;
}

int b200pt_set_frame_batch(b200pt_t* h, int n)
{
  if(!h || n < 1 || n > 64)
    return B200PT_E_INVALID;
  if(n == h->batch)
    return B200PT_OK;
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  h->batch = n;
  if(h->numPaths == 0)
    return B200PT_OK;
  float4* const user = (h->dAccum != h->dAccumOwned) ? h->dAccum : nullptr;
  int           rc;
  if(h->bandWorld > 1)
    rc = b200pt_resize_interleaved(h, h->width, h->height, h->bandRows, h->bandWorld, h->bandRank);
  else
    rc = b200pt_resize(h, h->width, h->height, h->tileY0, h->tileRows);
  if(rc == B200PT_OK && user)
    h->dAccum = user;
  return rc;
}

int b200pt_synchronize(b200pt_t* h)
{
  if(!h)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  return checkDeviceErrors(h);
}

int b200pt_set_profiling(b200pt_t* h, int enabled)
{
  if(!h)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  flushEvents(h);
  h->profiling = enabled != 0;
  if(h->profiling && h->evPool.empty())
  {
    h->evPool.resize(2048);
    for(auto& e : h->evPool)
    {
      CK(cudaEventCreate(&e.a));
      CK(cudaEventCreate(&e.b));
      e.cat = 3;
    }
  }
  return B200PT_OK;
}

int b200pt_render_frame(b200pt_t* h, const b200pt_frame_info* fi, const b200pt_push_constant* pc)
{
  if(!h || !fi || !pc)
    return B200PT_E_INVALID;
  if(!h->haveScene || h->numPaths == 0)
  {
    h->err = "b200pt_render_frame: set_scene and resize must come first";
    return B200PT_E_INVALID;
  }
  if(!(fi->flags & B200PT_SCENE_USE_HDR_ENVIRONMENT) || !h->haveEnv)
  {
    h->err = "b200pt_render_frame: only the HDR environment (--envSystem 1) is built; physical sky is out of scope";
    return B200PT_E_UNSUPPORTED;
  }
  if((fi->flags & B200PT_SCENE_USE_HDR_ENVIRONMENT) && fi->envBlur > 0.0f && !(fi->flags & B200PT_SCENE_USE_SOLID_BACKGROUND))
  {
    h->err = "b200pt_render_frame: the blurred HDR backplate (envBlur > 0: nvshaders' smoothHDRBlur, external) is not built";
    return B200PT_E_UNSUPPORTED;
  }
  if(pc->flags & B200PT_PT_USE_DLSS)
  {
    h->err = "b200pt_render_frame: the DLSS variant (frame jitter, motion vectors, specular guides) is out of scope";
    return B200PT_E_UNSUPPORTED;
  }
  if((pc->flags & B200PT_PT_USE_OPTIX_DENOISER) && !h->guides)
  {
    h->err = "b200pt_render_frame: ePtUseOptixDenoiser needs the guide image (b200pt_set_guide_outputs(h, 1) first)";
    return B200PT_E_INVALID;
  }
  if(pc->numSamples < 1 || pc->maxDepth < 0 || (int)fi->imageSize[0] != h->width || (int)fi->imageSize[1] != h->height)
  {
    h->err = "b200pt_render_frame: bad numSamples / maxDepth / imageSize";
    return B200PT_E_INVALID;
  }
  if(h->batch <= 1)
    return launchFrames(h, fi, pc, 1);
  // frame batching: collect consecutive frames of a static camera (same frame constants; push constants that differ only by
  // the frame / sample counters advancing like the host loop advances them) and run them as one wavefront
  if(h->pendingCount > 0)
  {
    const b200pt_push_constant& p0 = h->pendingPc;
    b200pt_push_constant        expect = p0;
    expect.frameCount = p0.frameCount + h->pendingCount;
    expect.totalSamples = p0.totalSamples + h->pendingCount * p0.numSamples;
    expect.flags = p0.flags & ~B200PT_PT_FIRST_FRAME;
    if(memcmp(&h->pendingFi, fi, sizeof(*fi)) != 0 || memcmp(&expect, pc, sizeof(*pc)) != 0)
    {
      const int rc = flushPending(h);
      if(rc)
        return rc;
    }
  }
  if(h->pendingCount == 0)
  {
    h->pendingFi = *fi;
    h->pendingPc = *pc;
  }
  h->pendingCount++;
  if(h->pendingCount >= h->batch)
    return flushPending(h);
  return B200PT_OK;
}

static int flushPending(b200pt_t* h)
{
  if(h->pendingCount == 0)
    return B200PT_OK;
  const int n = h->pendingCount;
  h->pendingCount = 0;
  return launchFrames(h, &h->pendingFi, &h->pendingPc, n);
}

int b200pt_flush(b200pt_t* h)
{
  if(!h)
    return B200PT_E_INVALID;
  return flushPending(h);
}

// enqueues the launch chain of `count` consecutive frames (count > 1: one batched wavefront, FrameParams::batch)
static int launchFrames(b200pt_t* h, const b200pt_frame_info* fi, const b200pt_push_constant* pc, int count)
{
  CK(cudaSetDevice(h->device));
  FrameParams F;
  F.fi = *fi;
  F.pc = *pc;
  F.width = h->width;
  F.height = h->height;
  F.tileY0 = h->tileY0;
  F.tileRows = h->tileRows;
  F.bandRows = h->bandRows;
  F.bandWorld = h->bandWorld;
  F.bandRank = h->bandRank;
  F.pixels = h->numPaths;
  F.batch = count;
  F.numPaths = h->numPaths * (uint32_t)count;

  const int     laneIdx = (int)(h->frameSerial++ % (uint64_t)h->numLanes);
  b200pt::Lane& L = h->lanes[laneIdx];
  cudaStream_t  st = L.stream;
  // the lane's pool is free once the accumulate of its previous frame ran; while profiling, frames are serialised
  // (wait for the previous frame's accumulate) so per-kernel event times are not inflated by overlap
  if(L.busy)
    CK(cudaStreamWaitEvent(st, L.freed, 0));
  if(h->profiling && h->lastLane >= 0 && h->lastLane != laneIdx)
    CK(cudaStreamWaitEvent(st, h->lanes[h->lastLane].freed, 0));
  uint32_t*    cntTrace = L.dCounters;             // [kMaxIters]
  uint32_t*    cntPost = L.dCounters + kMaxIters;  // [kMaxIters]
  uint32_t*    workTrace = L.dCounters + 2 * kMaxIters;  // dynamic-fetch cursors of the persistent kernels
  uint32_t*    workPost = L.dCounters + 3 * kMaxIters;
  uint32_t*    cntShadow = L.dCounters + 4 * kMaxIters;
  // any-hit counters of round r (r = 0: the main walk's candidates), continuation queue counters and cursors of round r, per ray kind
  constexpr int R = kContRounds;
  auto cntA = [&](int shadow, int r) { return L.dCounters + (size_t)(5 + shadow * (3 * R + 1) + r) * kMaxIters; };
  auto cntC = [&](int shadow, int r) { return L.dCounters + (size_t)(5 + shadow * (3 * R + 1) + (R + 1) + r) * kMaxIters; };
  auto wrkC = [&](int shadow, int r) { return L.dCounters + (size_t)(5 + shadow * (3 * R + 1) + (2 * R + 1) + r) * kMaxIters; };
  CK(cudaMemsetAsync(L.dCounters, 0, sizeof(uint32_t) * kCounterArrays * kMaxIters, st));

  enum
  {
    tTrace = 0,
    tShade = 1,
    tPost = 2,
    tOther = 3,
    tAnyHit = 4,
    tResolve = 5
  };
  const uint64_t frameNo = h->frameSerial - 1;
  auto timed = [&](int cat, auto&& launch) {
    if(h->profiling || h->timeline)
    {
      if(h->evUsed == h->evPool.size())
        flushEvents(h);
      b200pt::EvRec& r = h->evPool[h->evUsed++];
      r.cat = cat;
      r.lane = (st == h->stream) ? -1 : laneIdx;
      r.frame = frameNo;
      cudaEventRecord(r.a, st);
      launch();
      cudaEventRecord(r.b, st);
    }
    else
      launch();
    h->kernelLaunches++;
  };

  const int gridWide = gridFor(h, 8);
  timed(tOther, [&] { k_raygen<<<gridWide, 256, 0, st>>>(L.P, F, L.dQ[0], &cntTrace[0], h->dStats); });

  if(pc->maxDepth > 0)
  {
    int       it = 0;
    int       cur = 0;  // dQ[cur] = trace queue, dQ[2] = post queue, dQ[1-cur] = next queue
    const int firstBatch = pc->maxDepth;
    // (a shadowed shadow-catcher hit continues without consuming depth: such a frame can need more iterations than maxDepth)
    const bool catcherFrame = (fi->flags & B200PT_SCENE_USE_INFINITE_PLANE) && (fi->flags & B200PT_SCENE_INFINITE_PLANE_SHADOW_CATCHER);
    const bool mayOverrun = h->hasVolume || pc->numSamples > 1 || catcherFrame;
    int        remaining = firstBatch;
    for(;;)
    {
      for(int k = 0; k < remaining && it < kMaxIters - 1; k++, it++)
      {
        uint32_t* qT = L.dQ[cur];
        uint32_t* qN = L.dQ[1 - cur];
        // geometry walks are persistent kernels; the texture-dependent any-hit tests and the path bookkeeping run
        // as dense one-thread-per-path kernels (k_alpha, k_resolve) sized by the device-side queue counters
        const int gP = gridFor(h, 8);
        const int  gW = gridFor(h, 8);  // persistent walk kernels: 8 CTAs per SM, all resident (kTraceMinBlocks)
        // grids of the continuation rounds after the first: quarter-size below 8 M path slots.  Measured at N = 1 (20.7 M slots,
        // r02zj, one box): full 1021.1, quarter 1009.9 Mray/s.  On a 1/8 tile (2.6 M slots, r02fin2_n8 pass B) an almost empty
        // full-size walk launch costs about as much as the round saves in k_alpha; the quarter-size rule for such tiles follows
        // from that accounting and has NOT been measured at N > 1.
        const int  gSmall = F.numPaths < (8u << 20) ? gridFor(h, 2) : 0;  // 0: full grids
        const bool omm = h->S.bvh.ommRef != nullptr;  // scenes with opacity micromaps run the walk kernels' OMM instantiation
        const int gS = gridFor(h, 2);  // persistent shade kernel: 2 CTAs per SM (512-thread CTAs, one resident per SM)
        // geometry walks are persistent kernels; the texture-dependent any-hit tests and the path bookkeeping run
        // as dense kernels (k_alpha, k_resolve) sized by the device-side queue counters.  Any-hit: resolve kCand
        // candidates, one continuation round for the paths that used them all up, then whatever is still
        // undecided finishes inside the last k_alpha.
        timed(tTrace, [&] { WALK_KERNEL(k_trace, gW, L.P, h->S, qT, &cntTrace[it], &workTrace[it], L.dQ[4], cntA(0, 0) + it, h->dStats, kRefillThreshold, kPostponeShift, 0); });
        if(h->S.hasAlpha)
        {
          for(int r = 0; r < R; r++)
          {
            // rounds after the first see the few rays whose candidates were all rejected TWICE (about 1 % of the bounce); on small
            // wavefronts a quarter-size grid keeps the fixed cost of these extra launches down (see gSmall)
            const int gPr = (r && gSmall) ? gSmall : gP, gWr = (r && gSmall) ? gSmall : gW;
            timed(tAnyHit, [&] { k_alpha<false><<<gPr, 128, 2048, st>>>(L.P, h->S, L.dQ[4], cntA(0, r) + it, L.dQ[5], cntC(0, r) + it, h->dStats, r ? TRACE_CONT : 0); });
            timed(tTrace, [&] { WALK_KERNEL(k_trace, gWr, L.P, h->S, L.dQ[5], cntC(0, r) + it, wrkC(0, r) + it, L.dQ[4], cntA(0, r + 1) + it, h->dStats, kRefillThreshold, kPostponeShift, 1); });
          }
          timed(tAnyHit, [&] { k_alpha<false><<<gP, 128, 2048, st>>>(L.P, h->S, L.dQ[4], cntA(0, R) + it, nullptr, nullptr, h->dStats, TRACE_CONT); });
        }
        timed(tShade, [&] {
          if(h->featureMask == 0)
            k_shade<0u><<<gS, kShadeBlock, 2048, st>>>(L.P, h->S, F, qT, &cntTrace[it], L.dQ[2], &cntPost[it], L.dQ[3], &cntShadow[it], qN, &cntTrace[it + 1], h->dStats);
          else if(h->leanShade)
            k_shade<FEAT_LEAN><<<gS, kShadeBlock, 2048, st>>>(L.P, h->S, F, qT, &cntTrace[it], L.dQ[2], &cntPost[it], L.dQ[3], &cntShadow[it], qN, &cntTrace[it + 1], h->dStats);
          else
            k_shade<FEAT_ALL><<<gS, kShadeBlock, 2048, st>>>(L.P, h->S, F, qT, &cntTrace[it], L.dQ[2], &cntPost[it], L.dQ[3], &cntShadow[it], qN, &cntTrace[it + 1], h->dStats);
        });
        timed(tPost, [&] { WALK_KERNEL(k_shadow, gW, L.P, h->S, L.dQ[3], &cntShadow[it], &workPost[it], L.dQ[4], cntA(1, 0) + it, h->dStats, kRefillThreshold, kPostponeShift, 0); });
        if(h->S.hasAlpha)
        {
          for(int r = 0; r < R; r++)
          {
            const int gPr = (r && gSmall) ? gSmall : gP, gWr = (r && gSmall) ? gSmall : gW;
            timed(tAnyHit, [&] { k_alpha<true><<<gPr, 128, 2048, st>>>(L.P, h->S, L.dQ[4], cntA(1, r) + it, L.dQ[5], cntC(1, r) + it, h->dStats, r ? TRACE_CONT : 0); });
            timed(tPost, [&] { WALK_KERNEL(k_shadow, gWr, L.P, h->S, L.dQ[5], cntC(1, r) + it, wrkC(1, r) + it, L.dQ[4], cntA(1, r + 1) + it, h->dStats, kRefillThreshold, kPostponeShift, 1); });
          }
          timed(tAnyHit, [&] { k_alpha<true><<<gP, 128, 2048, st>>>(L.P, h->S, L.dQ[4], cntA(1, R) + it, nullptr, nullptr, h->dStats, TRACE_CONT); });
        }
        timed(tResolve, [&] { k_resolve<<<gridFor(h, 4), 256, 0, st>>>(L.P, h->S, F, L.dQ[2], &cntPost[it], qN, &cntTrace[it + 1], h->dStats); });
        cur = 1 - cur;
      }
      if(!mayOverrun)
        break;
      CK(cudaMemcpyAsync(L.hCount, &cntTrace[it], sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      if(L.hCount[0] == 0)
        break;
      if(it >= kMaxIters - 1)
      {
        h->err = "b200pt_render_frame: iteration budget exhausted (runaway volume walk?)";
        return B200PT_E_INVALID;
      }
      remaining = 4;
    }
  }
  else
  {
    // maxDepth == 0: every sample is black (the while loop never runs)
  }
  // accumulate on the main stream, in frame order
  CK(cudaEventRecord(L.done, st));
  CK(cudaStreamWaitEvent(h->stream, L.done, 0));
  st = h->stream;
  if(pc->flags & B200PT_PT_FIRST_FRAME)
    timed(tOther, [&] { k_select<<<gridFor(h, 8), 128, 0, st>>>(h->S, F, h->dSelect, h->dStats); });
  timed(tOther, [&] { k_accumulate<<<gridWide, 256, 0, st>>>(L.P, F, h->dAccum, h->dNdcDepth); });
  if((pc->flags & B200PT_PT_USE_OPTIX_DENOISER) && h->dGuide)
    timed(tOther, [&] { k_guide<<<gridWide, 256, 0, st>>>(L.P, F, h->dGuide); });
  CK(cudaEventRecord(L.freed, st));
  L.busy = true;
  h->lastLane = laneIdx;
  CK(cudaGetLastError());
  if(h->profiling && getenv("B200PT_DUMP_ITERS"))
  {
    // tuning aid: per-iteration queue sizes and kernel times of this frame (stderr)
    CK(cudaStreamSynchronize(st));
    const int            n = pc->maxDepth < 64 ? pc->maxDepth : 64;
    std::vector<uint32_t> c(2 * kMaxIters);
    CK(cudaMemcpy(c.data(), L.dCounters, sizeof(uint32_t) * 2 * kMaxIters, cudaMemcpyDeviceToHost));
    const size_t perIter = h->S.hasAlpha ? 11 : 5;
    const size_t first = h->evUsed >= perIter * (size_t)pc->maxDepth + 2 ? h->evUsed - (perIter * (size_t)pc->maxDepth + 2) : 0;
    for(int it = 0; it < n; it++)
    {
      float ms[6] = {0, 0, 0, 0, 0, 0};
      for(size_t k = 0; k < perIter; k++)
      {
        const size_t e = first + 1 + (size_t)it * perIter + k;
        float        t = 0.f;
        if(e < h->evUsed && cudaEventElapsedTime(&t, h->evPool[e].a, h->evPool[e].b) == cudaSuccess)
          ms[h->evPool[e].cat] += t;
      }
      fprintf(stderr, "iter %2d  %8u rays  k_trace %.3f  k_alpha %.3f  k_shade %.3f | %8u paths  k_shadow %.3f  k_resolve %.3f ms\n", it, c[it], ms[0], ms[4], ms[1],
              c[kMaxIters + it], ms[2], ms[5]);
    }
  }
  return B200PT_OK;
}

int b200pt_get_stats(b200pt_t* h, b200pt_stats* out)
{
  if(!h || !out)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  DevStats d{};
  CK(cudaMemcpy(&d, h->dStats, sizeof(d), cudaMemcpyDeviceToHost));
  out->closestRays = d.closestRays;
  out->shadowRays = d.shadowRays;
  out->shadedHits = d.shadedHits;
  out->pathsStarted = d.pathsStarted;
  out->nodesVisited = d.nodesVisited;
  out->trisTested = d.trisTested;
#ifdef B200PT_COUNT_TRAVERSAL
  if(getenv("B200PT_DUMP_ITERS") && d.warpIters)
    fprintf(stderr, "traversal loop: %llu warp iterations, busy lanes %.2f/32, node-phase lanes %.2f/32, triangle-phase lanes %.2f/32\n", d.warpIters,
            (double)d.busyLaneIters / (double)d.warpIters, (double)d.nodesVisited / (double)d.warpIters, (double)d.trisTested / (double)d.warpIters);
#endif
  flushEvents(h);
  out->msTraceClosest = h->msCat[0];
  out->msShade = h->msCat[1];
  out->msTraceShadow = h->msCat[2];
  out->msOther = h->msCat[3];
  out->msAnyHit = h->msCat[4];
  out->msResolve = h->msCat[5];
  out->launchesAnyHit = h->launchesCat[4];
  out->launchesResolve = h->launchesCat[5];
  out->msTotal = h->msCat[0] + h->msCat[1] + h->msCat[2] + h->msCat[3] + h->msCat[4] + h->msCat[5];
  out->kernelLaunches = h->kernelLaunches;
  out->launchesTraceClosest = h->launchesCat[0];
  out->launchesShade = h->launchesCat[1];
  out->launchesTraceShadow = h->launchesCat[2];
  return B200PT_OK;
}

int b200pt_reset_stats(b200pt_t* h)
{
  if(!h)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  {
    const int frc = flushPending(h);
    if(frc)
      return frc;
  }
  syncAll(h);
  CK(cudaMemset(h->dStats, 0, sizeof(DevStats)));
  flushEvents(h);
  for(int k = 0; k < 6; k++)
  {
    h->msCat[k] = 0;
    h->launchesCat[k] = 0;
  }
  h->kernelLaunches = 0;
  return B200PT_OK;
}

// ray-level API: the rays run through the production kernels on a scratch pool (round 1 had separate restart-per-candidate
// kernels here, so the ray-level parity tests did not cover the benchmarked code)
static int ensureRayPool(b200pt_t* h, uint32_t n)
{
  if(n <= h->rayCapacity)
    return B200PT_OK;
  syncAll(h);
  freeRayPool(h);
  int rc = allocPathState(h, h->rayAllocs, n, h->rayP);
  for(int k = 0; k < 3 && !rc; k++)
  {
    if(cudaMalloc((void**)&h->rayQ[k], (size_t)n * sizeof(uint32_t)) != cudaSuccess)
      rc = B200PT_E_NOMEM;
    else
      h->rayAllocs.push_back(h->rayQ[k]);
  }
  if(!rc)
  {
    if(cudaMalloc((void**)&h->rayCounters, 8 * sizeof(uint32_t)) != cudaSuccess)
      rc = B200PT_E_NOMEM;
    else
      h->rayAllocs.push_back(h->rayCounters);
  }
  if(rc)
  {
    cudaGetLastError();
    freeRayPool(h);
    h->err = "ray-level API: out of device memory";
    return rc;
  }
  h->rayCapacity = n;
  return B200PT_OK;
}

static int traceRays(b200pt_t* h, const float* dev_rays, uint32_t n, float* dev_out, uint32_t* dev_seeds, int shadow)
{
  if(!h || !h->haveScene || !dev_rays || !dev_out)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  if(n == 0)
    return B200PT_OK;
  const int rc = ensureRayPool(h, n);
  if(rc)
    return rc;
  cudaStream_t st = h->stream;
  PathState&   P = h->rayP;
  uint32_t*    c = h->rayCounters;  // [0] rays [1] any-hit [2] continuation [3] any-hit of the continuation [4..5] work cursors
  CK(cudaMemsetAsync(c, 0, 8 * sizeof(uint32_t), st));
  const int  gP = gridFor(h, 8);
  const bool omm = h->S.bvh.ommRef != nullptr;
  k_rays_load<<<gP, 256, 0, st>>>(P, reinterpret_cast<const float4*>(dev_rays), n, dev_seeds, h->rayQ[0], &c[0], shadow);
  if(!shadow)
  {
    WALK_KERNEL(k_trace, gP, P, h->S, h->rayQ[0], &c[0], &c[4], h->rayQ[1], &c[1], h->dStats, kRefillThreshold, kPostponeShift, TRACE_TMIN);
    if(h->S.hasAlpha)
    {
      k_alpha<false><<<gP, 128, 2048, st>>>(P, h->S, h->rayQ[1], &c[1], h->rayQ[2], &c[2], h->dStats, TRACE_TMIN);
      WALK_KERNEL(k_trace, gP, P, h->S, h->rayQ[2], &c[2], &c[5], h->rayQ[1], &c[3], h->dStats, kRefillThreshold, kPostponeShift, TRACE_TMIN | TRACE_CONT);
      k_alpha<false><<<gP, 128, 2048, st>>>(P, h->S, h->rayQ[1], &c[3], nullptr, nullptr, h->dStats, TRACE_TMIN | TRACE_CONT);
    }
  }
  else
  {
    WALK_KERNEL(k_shadow, gP, P, h->S, h->rayQ[0], &c[0], &c[4], h->rayQ[1], &c[1], h->dStats, kRefillThreshold, kPostponeShift, 0);
    if(h->S.hasAlpha)
    {
      k_alpha<true><<<gP, 128, 2048, st>>>(P, h->S, h->rayQ[1], &c[1], h->rayQ[2], &c[2], h->dStats, 0);
      WALK_KERNEL(k_shadow, gP, P, h->S, h->rayQ[2], &c[2], &c[5], h->rayQ[1], &c[3], h->dStats, kRefillThreshold, kPostponeShift, TRACE_CONT);
      k_alpha<true><<<gP, 128, 2048, st>>>(P, h->S, h->rayQ[1], &c[3], nullptr, nullptr, h->dStats, TRACE_CONT);
    }
  }
  k_rays_store<<<gP, 256, 0, st>>>(P, h->S, n, dev_out, dev_seeds, shadow);
  CK(cudaGetLastError());
  h->kernelLaunches += h->S.hasAlpha ? 6 : 3;
  return B200PT_OK;
}

int b200pt_trace_closest(b200pt_t* h, const float* dev_rays, uint32_t n, float* dev_hits, uint32_t* dev_seeds)
{
  return traceRays(h, dev_rays, n, dev_hits, dev_seeds, 0);
}

int b200pt_trace_shadow(b200pt_t* h, const float* dev_rays, uint32_t n, float* dev_transmission, uint32_t* dev_seeds)
{
  return traceRays(h, dev_rays, n, dev_transmission, dev_seeds, 1);
}

int b200pt_bsdf_eval(b200pt_t* h, const float* dev_in, uint32_t n, float* dev_out)
{
  if(!h || !dev_in || !dev_out)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  if(n)
    k_bsdf_eval<<<(n + 127) / 128, 128, 0, h->stream>>>(dev_in, n, dev_out);
  CK(cudaGetLastError());
  return B200PT_OK;
}

int b200pt_bsdf_sample(b200pt_t* h, const float* dev_in, uint32_t n, float* dev_out)
{
  if(!h || !dev_in || !dev_out)
    return B200PT_E_INVALID;
  CK(cudaSetDevice(h->device));
  if(n)
    k_bsdf_sample<<<(n + 127) / 128, 128, 0, h->stream>>>(dev_in, n, dev_out);
  CK(cudaGetLastError());
  return B200PT_OK;
}

}  // extern "C"
