// traverse.cuh — software traversal of the compressed 8-wide BVH (see bvh.h for the layout).
//
// Replaces the hardware TLAS/BLAS traversal behind RayQuery / TraceRay in the reference
// (shaders/raytracer_interface.h.slang:69-122 Trace, :139-187 TraceShadow).  One query primitive
// serves both: "closest hit whose (t, globalTriangleId) is lexicographically greater than a lower
// bound".  The any-hit loops of the reference (stochastic alpha, coloured transmission) become
// front-to-back iterations of that query, which makes the result independent of tree layout.
#pragma once
#include "bvh.h"
#include "omm.cuh"
#include "vec.cuh"

namespace pt {

struct TraceHit
{
  float    t;
  float    u, v;
  uint32_t slot;    // index into the triangle array, 0xFFFFFFFF = miss
  uint32_t gid;     // global (flatten-order) triangle id, tie-break key
  uint32_t w0;      // rnode | flags << 28
};

// one non-opaque candidate kept by a collecting traversal (see TravState::collectN)
struct Cand
{
  float    t, u, v;
  uint32_t slot, gid;
};
constexpr int kCand = 4;  // any-hit candidates kept per tree walk (k_alpha uses that many lanes per path)

struct BvhView
{
  const float4* __restrict__ nodes;  // 5 per node
  const float4* __restrict__ tris;   // 3 per triangle
  // opacity micromaps (omm.cuh): one reference word per triangle slot of THIS tree and the packed states; nullptr = the scene has none
  const uint32_t* __restrict__ ommRef = nullptr;
  const uint8_t* __restrict__ ommData = nullptr;
};

PT_D uint32_t extractByte(uint32_t x, int i) { return (x >> (i * 8)) & 0xffu; }
PT_D uint32_t signExtendS8x4(uint32_t x)
{
  // per byte: 0x80 -> 0xff, else 0x00  (vabsdiff4 trick replaced by plain bit math)
  return ((x >> 7) & 0x01010101u) * 0xffu;
}

// Byte J of x as a float WITHOUT the conversion unit and WITHOUT the ALU pipe.  History: 48 I2F.U8 per node saturated the XU
// pipe (r01); one PRMT per byte (byte into the mantissa of 2^15) moved the work to the ALU pipe, which then became the
// kernel's limiter (ncu r02c: pipe_alu 62 % of peak, issue 67 %, math_pipe_throttle; per child 14 ALU-pipe instructions against
// 7 on the FMA pipe).  tools/pipe_probe.cu on the B200: IDP.4A issues on the IMAD pipe, which overlaps BOTH the ALU pipe
// (PRMT / LOP3 / FMNMX) and the FFMA pipe.  So: dp4a(x, 64 << 8J, 0x48000000) adds b * 64 to the bit pattern of 2^17 = 131072.0f
// (mantissa ulp 2^-6), giving 131072 + b exactly, in one IMAD-pipe instruction.  The bias moves into the addend:
// t = (131072 + b) * ad + (ao - 131072 * ad); the addend's rounding error is at most |ad| / 128, the test widens by |ad| / 64.
constexpr float kByteBias = 131072.0f, kByteSlack = 0.015625f;
// byte J of x as an integer (SHF + LOP3 on the ALU pipe; doing these two extractions per child with IDP.4A as well was measured
// slower, 905 vs 944 Mray/s: the IMAD pipe then carries 64 instead of 48 instructions per node and becomes the longer one)
template <int J>
PT_D uint32_t extractByteJ(uint32_t x)
{
  return (x >> (8 * J)) & 0xffu;
}

template <int J>
PT_D float biasedByte(uint32_t x)
{
#ifdef __CUDA_ARCH__
  return __uint_as_float(__dp4a(x, 64u << (8 * J), 0x48000000u));
#else
  return __uint_as_float(0x48000000u + 64u * ((x >> (8 * J)) & 0xffu));
#endif
}

// (u, v) of a hit on a mirrored instance are stored swapped (the world-space winding was flipped at build time)
PT_D TraceHit unflipHit(TraceHit h)
{
  if(h.slot != 0xFFFFFFFFu && ((h.w0 >> 28) & TRI_FLIPPED))
  {
    const float u = h.u;
    h.u = h.v;
    h.v = u;
  }
  return h;
}

// rebuilds the traversal's record of an opaque hit from what the path state keeps of it (t, un-flipped u / v, slot)
PT_D TraceHit seedHit(const BvhView bvh, float t, float u, float v, uint32_t slot)
{
  TraceHit h;
  h.t = t;
  h.u = u;
  h.v = v;
  h.slot = slot;
  h.w0 = __float_as_uint(__ldg(&bvh.tris[slot * 3 + 0]).w);
  h.gid = __float_as_uint(__ldg(&bvh.tris[slot * 3 + 2]).w);
  return unflipHit(h);  // swapping twice restores the traversal-order (u, v)
}

// One traversal in flight, resumable one node-step at a time (the persistent kernels interleave the
// steps of 32 independent rays per warp and re-fill finished lanes from a global work counter).
//
// ONE tree holds every triangle; the per-triangle TRI_OPAQUE flag (getInstanceFlag, src/gltf_scene_rtx.cpp:271-295)
// decides what a geometric hit means, so a ray is ONE walk (round 1 walked an opaque tree and then an any-hit tree):
//   closest mode (IRaytracer::Trace, raytracer_interface.h.slang:69-122)
//     opaque hit      -> nearest-hit update of `best` in (t, global id) order
//     non-opaque hit  -> candidate for the stochastic alpha test: kept in a list of the kCand nearest ones, sorted by
//                        (t, id), if it lies in front of the opaque hit found so far
//     nodes are culled against bound = min(best.t, t of the kCand-th candidate once the list is full): every opaque
//     hit nearer than the last kept candidate is found (so candidates behind the true opaque hit can be dropped at
//     write-out and the list is then complete); when all kCand candidates lie in front, the any-hit kernel may reject
//     them all and a continuation walk resumes behind the last one -- it refines `best` as well.
//   shadow mode (IRaytracer::TraceShadow, :139-187, with the pinned order: any opaque occluder ends the query first)
//     opaque hit      -> done (occluded)
//     non-opaque hit  -> candidate list as above; the bound stays at the segment end (an occluder behind the kept
//                        candidates must still be found) unless the tree holds no opaque triangle (`shrink`).
//     Measured on the bench scene: shadow walks of the merged tree cost twice the round-1 pair of walks (opaque-only
//     tree with any-exit, then the any-hit tree with a shrinking bound: occluded rays never meet the foliage boxes), so
//     k_shadow keeps two trees and only k_trace walks the merged one.
//   cull    : back-face culling per triangle flags (RAY_FLAG_CULL_BACK_FACING_TRIANGLES + instance cull-disable)
//   lo      : only hits lexicographically after (loT, loId) in (t, global id) order count (continuation walks)
struct TravState
{
  const float4* nodes;
  const float4* tris;
  float3        org, dir;
  float         idx, idy, idz;
  float         tmin, tmax, tLow, loT, bound;
  uint32_t      loId, dsign;  // dsign: bit a set if the direction component along axis a (0 x, 1 y, 2 z) is >= 0
  bool          haveLo, cull, shadow, shrink;
  bool          overflow;  // a push found the stack full: the walk is incomplete (surfaced as a device error flag)
  TraceHit      best;
  uint2         cur;   // current node group (x = child base, y = hit bits << 24 | imask)
  uint2         tri;   // pending triangle group (x = triangle base, y = hit bits)
  int           sp;    // entries on the caller-provided stack (kept OUT of this struct so the rest stays in registers)
  int           collectN;  // candidates in the caller-provided list (sorted by (t, id))
#ifdef B200PT_COUNT_TRAVERSAL
  unsigned int nodeCount, triCount;
#endif

  PT_D void init(const BvhView bvh, float3 o, float3 d, float tmin_, float tmax_, bool cull_, bool shadow_, bool haveLo_, float loT_, uint32_t loId_,
                 bool shrink_ = true)
  {
    shrink = shrink_ || !shadow_;
    collectN = 0;
    nodes = bvh.nodes;
    tris = bvh.tris;
    org = o;
    dir = d;
    const float ooeps = 1e-20f;
    const float dx = fabsf(d.x) > ooeps ? d.x : copysignf(ooeps, d.x);
    const float dy = fabsf(d.y) > ooeps ? d.y : copysignf(ooeps, d.y);
    const float dz = fabsf(d.z) > ooeps ? d.z : copysignf(ooeps, d.z);
    idx = 1.0f / dx;
    idy = 1.0f / dy;
    idz = 1.0f / dz;
    dsign = (d.x < 0.f ? 0u : 1u) | (d.y < 0.f ? 0u : 2u) | (d.z < 0.f ? 0u : 4u);
    tmin = tmin_;
    tmax = tmax_;
    bound = tmax_;
    haveLo = haveLo_;
    loT = loT_;
    loId = loId_;
    tLow = haveLo_ ? fmaxf(tmin_, loT_) : tmin_;
    cull = cull_;
    shadow = shadow_;
    overflow = false;
    best.t = tmax_;
    best.slot = 0xFFFFFFFFu;
    best.gid = 0xFFFFFFFFu;
    best.u = best.v = 0.f;
    best.w0 = 0;
    cur = make_uint2(0u, 0x80000000u);
    tri = make_uint2(0u, 0u);
    sp = 0;
#ifdef B200PT_COUNT_TRAVERSAL
    nodeCount = triCount = 0;
#endif
  }

  // continuation walk: the opaque hit an earlier walk of the same ray found (an upper bound, possibly not yet the nearest)
  PT_D void seedOpaque(float t, float u, float v, uint32_t slot)
  {
    BvhView bv;
    bv.nodes = nodes;
    bv.tris = tris;
    best = seedHit(bv, t, u, v, slot);
    bound = fminf(bound, t);
  }

  static constexpr int kStackSize = 28;

  // One traversal step: (1) lanes without pending triangles open their next node, (2) lanes with pending
  // triangles test ONE triangle each — but only when enough lanes of the warp have one (vote); otherwise the
  // group is postponed onto the stack and node traversal continues (Ylitie et al. 2017, section 4.3).
  // Returns true when the traversal is complete.  `stack` is per-thread scratch of kStackSize entries (local memory),
  // `cand` the candidate list (entry i at cand[i * cs]: the kernels keep it in shared memory, one column per thread).
  // FORCE_OPAQUE: every triangle counts as opaque (IRaytracer::TraceLow, RAY_FLAG_FORCE_OPAQUE: the selection ray)
  // OMM: the scene carries opacity micromaps (a separate instantiation, so that scenes without them run the walk without the lookup)
  // MODE: the walk's protocol as a compile-time constant where the caller knows it (0 = the runtime flags of init(); 1 = closest-hit
  // walk: not a shadow query, back faces culled, the bound shrinks; 2 = shadow walk: shadow query, no culling) -- the per-triangle
  // flag tests and the shadow / closest branches fold away
  template <int KC = kCand, bool FORCE_OPAQUE = false, bool OMM = false, int MODE = 0>
  PT_D bool step(uint2* __restrict__ stack, int postponeShift, Cand* __restrict__ cand, int cs, const uint32_t* __restrict__ ommRef = nullptr,
                 const uint8_t* __restrict__ ommData = nullptr)
  {
    const bool shadow = MODE == 1 ? false : (MODE == 2 ? true : this->shadow);
    const bool cull = MODE == 1 ? true : (MODE == 2 ? false : this->cull);
    const bool shrink = MODE == 1 ? true : this->shrink;
    // single exit: an early return inside the divergent regions would move their reconvergence point out of the
    // caller's loop and the lanes of a warp would drift apart (measured: 8 of 32 lanes active)
    bool done = false;
    if(tri.y == 0)
    {
      if((cur.y & 0xff000000u) == 0)
      {
        if(sp == 0)
          done = true;
        else
          cur = stack[--sp];
      }
      if(done)
      {
      }
      else if(cur.y & 0xff000000u)
      {
        const uint32_t hitsImask = cur.y;
        const int      childBit = 31 - __clz(hitsImask);
        cur.y &= ~(1u << childBit);
        if(cur.y & 0xff000000u)
        {
          if(sp < kStackSize)
            stack[sp++] = cur;
          else
            overflow = true;
        }
        const uint32_t slotIndex = (uint32_t)(childBit - 24) ^ ((hitsImask >> 8) & 7u);  // the group carries its node's octant mask
        const uint32_t relative = __popc(hitsImask & ~(0xffffffffu << slotIndex));
        const uint32_t nodeIndex = cur.x + relative;
#ifdef B200PT_COUNT_TRAVERSAL
        nodeCount++;
#endif
        const float4 n0 = __ldg(&nodes[nodeIndex * 5 + 0]);
        const float4 n1 = __ldg(&nodes[nodeIndex * 5 + 1]);
        const float4 n2 = __ldg(&nodes[nodeIndex * 5 + 2]);
        const float4 n3 = __ldg(&nodes[nodeIndex * 5 + 3]);
        const float4 n4 = __ldg(&nodes[nodeIndex * 5 + 4]);

        const uint32_t eImask = __float_as_uint(n0.w);
        const float    adx = __uint_as_float(extractByte(eImask, 0) << 23) * idx;
        const float    ady = __uint_as_float(extractByte(eImask, 1) << 23) * idy;
        const float    adz = __uint_as_float(extractByte(eImask, 2) << 23) * idz;
        // quantised plane bytes -> floats with the bias folded into the addend, conservative slack (see biasedByte)
        const float aox = fmaf(-kByteBias, adx, (n0.x - org.x) * idx);
        const float aoy = fmaf(-kByteBias, ady, (n0.y - org.y) * idy);
        const float aoz = fmaf(-kByteBias, adz, (n0.z - org.z) * idz);
        const float aoxN = fmaf(-kByteSlack, fabsf(adx), aox), aoxF = fmaf(kByteSlack, fabsf(adx), aox);
        const float aoyN = fmaf(-kByteSlack, fabsf(ady), aoy), aoyF = fmaf(kByteSlack, fabsf(ady), aoy);
        const float aozN = fmaf(-kByteSlack, fabsf(adz), aoz), aozF = fmaf(kByteSlack, fabsf(adz), aoz);

        // per-node axis map (bvh.cpp): bit k of the node's octant mask is the direction sign along the axis slot bit k follows
        const uint32_t n1x = __float_as_uint(n1.x);
        const uint32_t amap = n1x >> 26;
        const uint32_t octN = ((dsign >> (amap & 3u)) & 1u) | (((dsign >> ((amap >> 2) & 3u)) & 1u) << 1) | (((dsign >> (amap >> 4)) & 1u) << 2);
        const uint32_t octInv4 = octN * 0x01010101u;
        cur.x = n1x & 0x03ffffffu;
        tri.x = __float_as_uint(n1.y);

        uint32_t hitMask = 0;
#pragma unroll
        for(int i = 0; i < 2; i++)
        {
          const uint32_t meta4 = __float_as_uint(i == 0 ? n1.z : n1.w);
          const uint32_t isInner4 = (meta4 & (meta4 << 1)) & 0x10101010u;
          const uint32_t innerMask4 = signExtendS8x4(isInner4 << 3);
          const uint32_t bitIndex4 = (meta4 ^ (octInv4 & innerMask4)) & 0x1f1f1f1fu;
          const uint32_t childBits4 = (meta4 >> 5) & 0x07070707u;

          const uint32_t qlox = __float_as_uint(i == 0 ? n2.x : n2.y), qhix = __float_as_uint(i == 0 ? n2.z : n2.w);
          const uint32_t qloy = __float_as_uint(i == 0 ? n3.x : n3.y), qhiy = __float_as_uint(i == 0 ? n3.z : n3.w);
          const uint32_t qloz = __float_as_uint(i == 0 ? n4.x : n4.y), qhiz = __float_as_uint(i == 0 ? n4.z : n4.w);
          const uint32_t xmin = dir.x < 0.f ? qhix : qlox, xmax = dir.x < 0.f ? qlox : qhix;
          const uint32_t ymin = dir.y < 0.f ? qhiy : qloy, ymax = dir.y < 0.f ? qloy : qhiy;
          const uint32_t zmin = dir.z < 0.f ? qhiz : qloz, zmax = dir.z < 0.f ? qloz : qhiz;
#define PT_CHILD(J)                                                                                                        \
  {                                                                                                                        \
    const float tminx = fmaf(biasedByte<J>(xmin), adx, aoxN);                                                              \
    const float tminy = fmaf(biasedByte<J>(ymin), ady, aoyN);                                                              \
    const float tminz = fmaf(biasedByte<J>(zmin), adz, aozN);                                                              \
    const float tmaxx = fmaf(biasedByte<J>(xmax), adx, aoxF);                                                              \
    const float tmaxy = fmaf(biasedByte<J>(ymax), ady, aoyF);                                                              \
    const float tmaxz = fmaf(biasedByte<J>(zmax), adz, aozF);                                                              \
    const float tn = fmaxf(fmaxf(tminx, tminy), fmaxf(tminz, tLow));                                                       \
    const float tf = fminf(fminf(tmaxx, tmaxy), fminf(tmaxz, bound));                                                      \
    /* widen by a few ulp: keeps the box test conservative w.r.t. the triangle test */                                     \
    const bool     in = tn <= tf * 1.000001f;                                                                              \
    const uint32_t childBits = in ? extractByteJ<J>(childBits4) : 0u;                                                      \
    hitMask |= childBits << extractByteJ<J>(bitIndex4);                                                                    \
  }
          PT_CHILD(0)
          PT_CHILD(1)
          PT_CHILD(2)
          PT_CHILD(3)
#undef PT_CHILD
        }
        cur.y = (hitMask & 0xff000000u) | (octN << 8) | (eImask >> 24);
        tri.y = hitMask & 0x00ffffffu;
      }
      else
      {
        // a postponed triangle group came off the stack
        tri = cur;
        cur = make_uint2(0u, 0u);
      }
    }

    // ---- triangle phase (one triangle per lane per step) ------------------------------------------------
    const unsigned conv = __activemask();
    const unsigned haveTri = __ballot_sync(conv, !done && tri.y != 0);
    if(!done && tri.y != 0)
    {
      // postpone when few lanes would take part and this lane's current node group still has children to open
      // (the group goes under the next node; `cur` only ever holds node groups)
      if((__popc(haveTri) << postponeShift) < __popc(conv) && (cur.y & 0xff000000u) != 0 && sp < kStackSize)
      {
        stack[sp++] = tri;
        tri.y = 0;
      }
      else
      {
        const int triBit = 31 - __clz(tri.y);
        tri.y &= ~(1u << triBit);
        const uint32_t slot = tri.x + (uint32_t)triBit;
#ifdef B200PT_COUNT_TRAVERSAL
        triCount++;
#endif
        const float4 a = __ldg(&tris[slot * 3 + 0]);
        const float4 b = __ldg(&tris[slot * 3 + 1]);
        const float4 c = __ldg(&tris[slot * 3 + 2]);
        const float3 v0 = f3(a.x, a.y, a.z), e1 = f3(b.x, b.y, b.z), e2 = f3(c.x, c.y, c.z);
        // Moeller-Trumbore, explicit fma chain (bit-identical to oracle/pt_oracle.cpp intersectTri); branch-free
        // up to the final update so the lanes stay converged
        const float3   pvec = crossFma(dir, e2);
        const float    det = dotFma(e1, pvec);
        const float    inv = 1.0f / det;
        const float3   tvec = org - v0;
        const float    u = dotFma(tvec, pvec) * inv;
        const float3   qvec = crossFma(tvec, e1);
        const float    v = dotFma(dir, qvec) * inv;
        const float    t = dotFma(e2, qvec) * inv;
        const uint32_t w0 = __float_as_uint(a.w);
        const uint32_t flags = w0 >> 28;
        const uint32_t gid = __float_as_uint(c.w);
        bool           hit = (det != 0.0f) & (u >= 0.0f) & (u <= 1.0f) & (v >= 0.0f) & (u + v <= 1.0f) & (t > tmin) & (t < tmax);
        const bool     front = (flags & TRI_FLIPPED) ? (det < 0.0f) : (det > 0.0f);
        hit &= !cull | ((flags & TRI_NOCULL) != 0) | front;
        hit &= !haveLo | (t > loT) | ((t == loT) & (gid > loId));
        bool opq = FORCE_OPAQUE || (flags & TRI_OPAQUE) != 0;
        if(OMM && !FORCE_OPAQUE && hit && !opq && ommRef != nullptr)
        {
          // what the RT cores do with an opacity micromap: the micro-triangle under the hit decides -- OPAQUE is committed like a
          // FORCE_OPAQUE triangle, TRANSPARENT is culled, only UNKNOWN becomes an any-hit candidate (omm.cuh)
          const bool fl = (flags & TRI_FLIPPED) != 0;  // mirrored instance: the record's 2nd / 3rd vertex are swapped
          const int  st = ommStateOf(__ldg(&ommRef[slot]), fl ? v : u, fl ? u : v, [&](uint32_t o) { return (uint32_t)__ldg(&ommData[o]); });
          opq = st == OMM_OPAQUE;
          hit = st != OMM_TRANSPARENT;
        }
        if(hit)
        {
          if(opq)
          {
            if((t < best.t) | ((t == best.t) & (gid < best.gid)))
            {
              best.t = t;
              best.u = u;
              best.v = v;
              best.slot = slot;
              best.gid = gid;
              best.w0 = w0;
              if(shadow)
                done = true;  // occlusion query satisfied
              else
                bound = fminf(bound, t);
            }
          }
          else
          {
            // candidate for the any-hit kernel: in front of the opaque hit (closest mode) and, once the list is full,
            // in front of its last entry
            bool keep = shadow | (t < best.t);
            if(collectN == KC)
            {
              const float    lt = cand[(KC - 1) * cs].t;
              const uint32_t lg = cand[(KC - 1) * cs].gid;
              keep &= (t < lt) | ((t == lt) & (gid < lg));
            }
            if(keep)
            {
              // insertion sort by (t, id); a full list drops its last entry
              int pos = collectN < KC ? collectN : KC - 1;
              while(pos > 0)
              {
                const Cand p = cand[(pos - 1) * cs];
                if(!((p.t > t) | ((p.t == t) & (p.gid > gid))))
                  break;
                cand[pos * cs] = p;
                pos--;
              }
              Cand nc;
              nc.t = t;
              nc.u = u;
              nc.v = v;
              nc.slot = slot;
              nc.gid = gid;
              cand[pos * cs] = nc;
              if(collectN < KC)
                collectN++;
              if(collectN == KC && shrink)
                bound = fminf(bound, cand[(KC - 1) * cs].t);
            }
          }
        }
      }
    }
    return done | ((tri.y == 0) & ((cur.y & 0xff000000u) == 0) & (sp == 0));
  }

  // the opaque hit with (u,v) restored for mirrored instances
  PT_D TraceHit result() const { return unflipHit(best); }

  // closest mode: candidates in front of the opaque hit (the list is sorted, so a prefix of it)
  PT_D int candidatesInFront(const Cand* __restrict__ cand, int cs) const
  {
    int n = 0;
    while(n < collectN && (best.slot == 0xFFFFFFFFu || cand[n * cs].t < best.t))
      n++;
    return n;
  }

  PT_D void flushCounters(unsigned long long* nodeCounter, unsigned long long* triCounter)
  {
#ifdef B200PT_COUNT_TRAVERSAL
    if(nodeCounter)
      atomicAdd(nodeCounter, (unsigned long long)nodeCount);
    if(triCounter)
      atomicAdd(triCounter, (unsigned long long)triCount);
    nodeCount = triCount = 0;
#else
    (void)nodeCounter;
    (void)triCounter;
#endif
  }
};

// One complete walk on one lane (the any-hit kernels' rare in-kernel fallback; the host-side check of this source):
// the up-to-KC nearest candidates behind the lower bound, sorted, in `cand`; `opq` carries the opaque hit in and out
// (closest mode: refined; shadow mode: slot != miss means occluded).  Returns the number of candidates that count
// (closest mode: those in front of the opaque hit).  *overflowed is OR-ed with the stack-overflow flag.
template <int KC = kCand>
PT_D int walkCollect(const BvhView bvh, float3 org, float3 dir, float tmin, float tmax, bool cull, bool shadow, bool shrink, bool haveLo, float loT, uint32_t loId,
                     TraceHit& opq, Cand* __restrict__ cand, bool* overflowed = nullptr, int* deepest = nullptr)
{
  TravState T;
  uint2     stack[TravState::kStackSize];
  T.init(bvh, org, dir, tmin, tmax, cull, shadow, haveLo, loT, loId, shrink);
  if(opq.slot != 0xFFFFFFFFu)
  {
    T.best = opq;
    T.bound = fminf(T.bound, opq.t);
  }
  while(!T.template step<KC, false, true>(stack, 2, cand, 1, bvh.ommRef, bvh.ommData))
  {
    if(deepest && T.sp > *deepest)
      *deepest = T.sp;
  }
  if(overflowed && T.overflow)
    *overflowed = true;
  opq = T.best;
  return shadow ? T.collectN : T.candidatesInFront(cand, 1);
}

}  // namespace pt
