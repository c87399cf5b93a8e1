// device_scene.cuh — HBM-resident scene + per-frame parameter blocks shared by all kernels.
//
// Data contract = what SceneVk / MaterialCache / HdrIbl give the reference shaders
// (shaders/gltf_scene_io.h.slang:41-322; shaders/shaderio.h:148-196), re-laid for CUDA:
//   GltfRenderNode[] / GltfShadeMaterial[] / GltfTextureInfo[] / GltfLight[]  : same bytes, AoS
//   GltfRenderPrimitive (7 device addresses)                                  : DevPrim
//   bindless Sampler2D allTextures[]                                          : cudaTextureObject_t[]
//   HDR env Sampler2D + StructuredBuffer<EnvAccel>                            : float4[] + uint2[]
//   TLAS/BLAS                                                                 : BvhView (+ triMeta)
#pragma once
#include <cuda_runtime.h>

#include "../../include/b200pt.h"
#include "traverse.cuh"

namespace pt {

struct DevPrim
{
  const uint32_t* idx;
  const float*    pos;
  const float*    nrm;
  const uint32_t* col;
  const float*    tan;
  const float*    uv0;
  const float*    uv1;
};

struct DevTex
{
  // RGBA8 mip pyramid in plain global memory, every level stored as 4x4-texel tiles (64 B: a bilinear footprint
  // mostly stays inside one tile).  Filtering happens in fp32 in the kernel, so the texture unit would only ever
  // point-sample -- and with one texture object per lane every TEX became a waterfall loop over the distinct
  // handles in the warp (SASS: R2UR + BRA.U.ANY around each of the 24 fetches of a shaded hit).
  const uchar4*   texels;
  const uint32_t* levelOfs;  // texel offset of every level from `texels`
  int             w0, h0;
  float           maxLevel;
  int             wrapS, wrapT;  // glTF enums
  int             srgb;
  int             magLinear, minLinear, mipLinear;
};

// Everything the stochastic alpha test of ONE non-opaque triangle needs (getOpacity, pathtrace_functions.h.slang:189-260),
// gathered at scene build: 64 B = four 128-bit loads, against the nine dependent gathers of the generic path (candidate ->
// triMeta -> render node -> primitive -> indices -> uv -> material -> texture info -> texture descriptor) that made the
// any-hit kernels latency-bound (ncu r01: long_scoreboard 20-27 warps per issue).
struct AlphaRec
{
  float         uv[6];        // the three vertices' texture coordinates of the set the alpha texture reads ((0,0) if absent)
  const uchar4* lv0;          // level-0 texels of the base-colour / diffuse texture (tiled), nullptr = no texture (alpha 1)
  int           w0, h0;
  uint32_t      wrap;         // wrapS | wrapT << 16 (glTF enums)
  float         factor;       // pbrBaseColorFactor.a (pbrDiffuseFactor.a for specular-glossiness)
  float         cutoff;
  uint32_t      modeFlags;    // bits 0-1 alphaMode, bit 2 magnification filter is linear, bit 3 vertex colours present
  uint32_t      colA;         // vertex colour alphas: a0 | a1 << 8 | a2 << 16 (UNORM8)
  float         transmission; // material.transmissionFactor (<= 0.01: a passing candidate blocks the shadow ray)
};
static_assert(sizeof(AlphaRec) == 64, "AlphaRec is four 16-byte loads");

// The vertex attributes of ONE triangle of a render primitive, gathered at scene build (object space, shared by all
// instances of the primitive): twelve 128-bit loads instead of the dependent chain index -> 3 vertices x {position, normal,
// uv0, uv1, colour, tangent} of narrow loads that getHitState (get_hit.h.slang:59-173) otherwise walks.
struct ShadeRec
{
  // twelve float4, laid out so that every attribute is read by named components (no address arithmetic on the device):
  //   v[0] = pos0.xyz | flags      v[1] = pos1.xyz | col0     v[2] = pos2.xyz | col1     v[3] = nrm0.xyz | col2
  //   v[4] = nrm1.xyz | uv0[0].x   v[5] = nrm2.xyz | uv0[0].y v[6] = uv0[1].xy, uv0[2].xy
  //   v[7] = uv1[0].xy, uv1[1].xy  v[8] = uv1[2].xy | 0 | 0   v[9..11] = tangent 0..2 (xyzw)
  // flags: bit 0 normals, 1 uv0, 2 uv1, 3 colours, 4 tangents present (else the reference's fallbacks apply)
  float4 v[12];
};
static_assert(sizeof(ShadeRec) == 192, "ShadeRec is twelve 16-byte loads");

struct DevScene
{
  const b200pt_render_node*    nodes;
  const DevPrim*               prims;
  const b200pt_shade_material* mats;
  const b200pt_texture_info*   texInfos;
  const DevTex*                textures;
  const b200pt_light*          lights;
  int                          numLights;
  int                          numTextures;
  BvhView                      bvh;       // closest-hit walks: ONE tree over every triangle; TRI_OPAQUE per triangle decides hit vs candidate
  BvhView                      bvhO;      // shadow walks, phase 0: FORCE_OPAQUE triangles only (any hit ends the query)
  BvhView                      bvhA;      // shadow walks, phase 1: non-opaque triangles only (candidates); shares bvhO's triangle array
  int                          hasAlpha;  // the scene has non-opaque triangles (the any-hit kernels are launched)
  const uint2*                 triMeta;   // per triangle slot of `bvh`: (rnode | flags<<28, primitiveID)
  const uint2*                 triMetaS;  // per triangle slot of bvhO / bvhA (== triMeta in scenes without non-opaque triangles)
  int                          numMaterials;
  const ShadeRec*              shadeRecs; // one per triangle of every render primitive
  const uint32_t*              shadeIdx;  // per triangle slot of `bvh`: index into shadeRecs
  const AlphaRec*              alphaRecs; // one per non-opaque triangle, in bvhA's leaf order
  const uint32_t*              alphaIdx;  // per triangle slot of `bvh`: index into alphaRecs (0xFFFFFFFF for opaque triangles)
  uint32_t                     alphaBaseS; // first non-opaque slot of the split triangle array: record = slot - alphaBaseS
  const float4*                envRgba;  // lat-long radiance, pdf in .w
  const uint2*                 envAccel; // (alias, q bits)
  const float*                 lutSrgb;  // 512 floats: sRGB decode table, then i/255 (staged into shared memory per block)
  int                          envW, envH;
};

struct FrameParams
{
  b200pt_frame_info    fi;
  b200pt_push_constant pc;
  int                  width, height;
  int                  tileY0, tileRows;
  int                  bandRows, bandWorld, bandRank;  // interleaved tiles: bandWorld > 1 (then tileY0 == 0)
  uint32_t             numPaths;  // path slots of this launch chain = pixels * batch
  // Frame batching (b200pt_set_frame_batch): `batch` consecutive frames of a static camera run as ONE wavefront.  Slot i
  // belongs to pixel i % pixels of frame pc.frameCount + i / pixels; pc holds the FIRST frame's constants, frame b adds b to
  // frameCount and b * numSamples to totalSamples (what the host loop would have passed, src/renderer_pathtracer.cpp:1496-1574).
  uint32_t             pixels;    // tileRows * width
  int                  batch;     // >= 1
};

PT_D uint32_t pixelOf(const FrameParams& F, uint32_t i) { return F.batch > 1 ? i % F.pixels : i; }
PT_D uint32_t frameOf(const FrameParams& F, uint32_t i) { return F.batch > 1 ? i / F.pixels : 0u; }
// the slot renders the first frame of an accumulation (its sample overwrites the image, frame-0 outputs are written)
PT_D bool isFirstFrame(const FrameParams& F, uint32_t i) { return (F.pc.flags & B200PT_PT_FIRST_FRAME) != 0 && (F.batch <= 1 || i < F.pixels); }

// global pixel row of tile pixel p (seeds always use global coordinates)
PT_D uint32_t pixelRow(const FrameParams& F, uint32_t p)
{
  const uint32_t l = p / (uint32_t)F.width;
  if(F.bandWorld <= 1)
    return (uint32_t)F.tileY0 + l;
  return ((l / (uint32_t)F.bandRows) * (uint32_t)F.bandWorld + (uint32_t)F.bandRank) * (uint32_t)F.bandRows + l % (uint32_t)F.bandRows;
}

// ---- wavefront path state (SoA, one slot per pixel of the tile) --------------------------------
// 16-byte records so every access is one 128-bit load/store.
struct PathState
{
  float4*   rayO;    // origin.xyz | cone width
  float4*   rayD;    // direction.xyz | tmax
  float4*   hit;     // t | u | v | triangle slot (bits; 0xFFFFFFFF = miss)
  float4*   thr;     // throughput.xyz | lastSamplePdf
  float4*   rad;     // radiance.xyz | scatterBounces (bits)
  float4*   misc;    // maxRoughness.xy | flags (bits) | seed (bits)
  uint4*    medium;  // fp16x3 extinction | fp16x3 scatter | fp16 anisotropy (packed) | sample index
  float4*   pixSum;  // per-pixel sum of the frame's samples (rgb + solid flag)
  float4*   shO;     // shadow ray origin.xyz | tmax
  float4*   shD;     // shadow ray direction.xyz | unused
  float4*   shC;     // NEE contribution.xyz | unused
  float4*   firstHit;  // first frame only: world position of the sample's first surface hit | 1 (primary miss: direction | 0)
  // any-hit candidates of the ray last traced for the path (closest-hit ray, then the shadow ray): up to kCand
  // nearest non-opaque hits as t | u | v | triangle slot, written by the traversal kernels and consumed by the
  // dense alpha / resolve kernels
  float4*   cand[kCand];
  uint2*    candInfo;  // x: count (bit 31: an opaque occluder ended the shadow query) | y: global id of the last candidate
  // denoiser guides of the sample's first hit (GuideScratch, pathtrace_functions.h.slang:79-88; null unless b200pt_set_guide_outputs):
  // albedo.xyz | roughness and normal.xyz | 1 (0: the primary ray missed), every value rounded through fp16 like the reference's float16_t fields
  float4*   guideA;
  float4*   guideN;
};

// flags word in misc.z
enum : uint32_t
{
  PF_DEPTH_MASK = 0xffffu,
  PF_INSIDE = 1u << 16,
  PF_SOLID = 1u << 17,
  PF_POST_VOLUME = 1u << 18,   // post stage runs the in-volume RR rule instead of the surface one
  PF_SHADOW_VALID = 1u << 19,
  PF_SHADOW_INSIDE = 1u << 20, // TraceShadow(initialInside = true)
  PF_CATCHER = 1u << 21,       // the path sits on the shadow-catcher plane: the post stage runs handleShadowCatcher's second half
};

struct Queues
{
  uint32_t* qTrace;   // paths to trace + shade this iteration
  uint32_t* qPost;    // paths entering the shadow / RR stage
  uint32_t* qNext;    // paths for the next iteration
  uint32_t* counters; // [0] = count(qTrace) [1] = count(qPost) [2] = count(qNext)
};

struct DevStats
{
  unsigned long long closestRays, shadowRays, shadedHits, pathsStarted, nodesVisited, trisTested;
  unsigned long long warpIters, busyLaneIters;  // counter build only: traversal-loop iterations per warp, busy lanes summed
  unsigned long long errorFlags;                // bit 0: a traversal stack overflowed (the walk was incomplete)
};

}  // namespace pt
