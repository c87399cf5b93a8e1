// shade.cuh — device functions of the shade / shadow stages: hit-attribute fetch, glTF material
// evaluation with bindless textures, environment + punctual light sampling, volumes.
//
// Restates, stage by stage (reference file:line):
//   getHitState                          shaders/get_hit.h.slang:59-173
//   evaluateMaterial / getTexture        shaders/gltf_material_eval.h.slang:76-457
//   getOpacity / getShadowTransmission   shaders/pathtrace_functions.h.slang:189-343
//   sampleLights / sampleEnvironment     shaders/pathtrace_functions.h.slang:357-492
//   volume medium + scatter              shaders/pathtrace_functions.h.slang:118-140, 605-672
#pragma once
#include <cuda_fp16.h>

#include "bsdf.cuh"
#include "device_scene.cuh"

namespace pt {

// ---- vertex access (shaders/gltf_vertex_access.h.slang) -----------------------------------------
PT_D float3 ld3(const float* a, uint32_t i) { return f3(__ldg(a + i * 3), __ldg(a + i * 3 + 1), __ldg(a + i * 3 + 2)); }
PT_D float2 ld2(const float* a, uint32_t i)
{
  const float2 v = __ldg(reinterpret_cast<const float2*>(a) + i);
  return v;
}
PT_D float4 ld4(const float* a, uint32_t i) { return __ldg(reinterpret_cast<const float4*>(a) + i); }
PT_D float4 unpackUnorm4x8(uint32_t p)
{
  return f4((float)((p >> 0) & 0xFF) / 255.0f, (float)((p >> 8) & 0xFF) / 255.0f, (float)((p >> 16) & 0xFF) / 255.0f, (float)((p >> 24) & 0xFF) / 255.0f);
}
PT_D float2 interpTexCoord(const DevPrim& P, int channel, uint3 tri, float3 bary)
{
  const float* uv = channel ? P.uv1 : P.uv0;
  if(uv == nullptr)
    return f2(0.0f, 0.0f);
  return ld2(uv, tri.x) * bary.x + ld2(uv, tri.y) * bary.y + ld2(uv, tri.z) * bary.z;
}
PT_D float4 interpColor(const DevPrim& P, uint3 tri, float3 bary)
{
  if(P.col == nullptr)
    return f4(1, 1, 1, 1);
  return unpackUnorm4x8(__ldg(P.col + tri.x)) * bary.x + unpackUnorm4x8(__ldg(P.col + tri.y)) * bary.y + unpackUnorm4x8(__ldg(P.col + tri.z)) * bary.z;
}
PT_D uint3 loadTri(const DevPrim& P, uint32_t t) { return make_uint3(__ldg(P.idx + t * 3), __ldg(P.idx + t * 3 + 1), __ldg(P.idx + t * 3 + 2)); }

// ---- hit state ----------------------------------------------------------------------------------
struct HitState
{
  float3 pos, nrm;
  float4 color;
  float3 geonrm, shadowPos;
  float2 uv0, uv1;
  float3 tangent, bitangent;
  float  texelDensity;
};

PT_D ShadeRec loadShadeRec(const ShadeRec* __restrict__ p)
{
  const float4* q = reinterpret_cast<const float4*>(p);
  ShadeRec      r;
#pragma unroll
  for(int i = 0; i < 12; i++)
    r.v[i] = __ldg(q + i);
  return r;
}

// getHitState (get_hit.h.slang:59-173) on the triangle's pre-gathered attribute record: the arithmetic is the reference's,
// statement by statement; only where the vertex data comes from differs (device_scene.cuh: ShadeRec)
PT_D HitState getHitState(const ShadeRec& R, float3 bary, const float* W2O, const float* O2W, float3 rayDir)
{
  HitState       hit;
  const uint32_t flags = __float_as_uint(R.v[0].w);
  const bool     hasNrm = (flags & 1u) != 0, hasUv0 = (flags & 2u) != 0, hasUv1 = (flags & 4u) != 0, hasCol = (flags & 8u) != 0, hasTan = (flags & 16u) != 0;
  const float3   pos0 = xyz(R.v[0]), pos1 = xyz(R.v[1]), pos2 = xyz(R.v[2]);
  const float3 position = pos0 * bary.x + pos1 * bary.y + pos2 * bary.z;
  hit.pos = xfPoint(O2W, position);

  const float3 geoNormal = normalize(cross(pos1 - pos0, pos2 - pos0));
  hit.geonrm = normalize(xfNormal(W2O, geoNormal));

  float3 nrm0 = geoNormal, nrm1 = geoNormal, nrm2 = geoNormal, normal = geoNormal;
  if(hasNrm)
  {
    nrm0 = xyz(R.v[3]);
    nrm1 = xyz(R.v[4]);
    nrm2 = xyz(R.v[5]);
    normal = nrm0 * bary.x + nrm1 * bary.y + nrm2 * bary.z;
  }
  hit.nrm = normalize(xfNormal(W2O, normal));

  const bool  frontFace = dot(hit.geonrm, rayDir) < 0.0f;
  const float sideFlip = frontFace ? 1.0f : -1.0f;
  // shadow-terminator offset (Hanika 2021), get_hit.h.slang:102-106
  const float3 shadowPos = pointOffset(position, pos0, pos1, pos2, nrm0 * sideFlip, nrm1 * sideFlip, nrm2 * sideFlip, bary);
  hit.shadowPos = xfPoint(O2W, shadowPos);

  const float2 t0 = f2(R.v[4].w, R.v[5].w), t1 = f2(R.v[6].x, R.v[6].y), t2 = f2(R.v[6].z, R.v[6].w);
  hit.uv0 = hasUv0 ? t0 * bary.x + t1 * bary.y + t2 * bary.z : f2(0.0f, 0.0f);
  hit.uv1 = hasUv1 ? f2(R.v[7].x, R.v[7].y) * bary.x + f2(R.v[7].z, R.v[7].w) * bary.y + f2(R.v[8].x, R.v[8].y) * bary.z : f2(0.0f, 0.0f);
  if(hasUv0)
  {
    const float3 we1 = xfVector(O2W, pos1 - pos0);
    const float3 we2 = xfVector(O2W, pos2 - pos0);
    const float  wArea = length(cross(we1, we2));
    const float2 duv1 = t1 - t0, duv2 = t2 - t0;
    const float  uvArea = fabsf(duv1.x * duv2.y - duv1.y * duv2.x);
    hit.texelDensity = sqrtf(fmaxf(uvArea, 1e-20f) / fmaxf(wArea, 1e-20f));
  }
  else
    hit.texelDensity = 0.0f;

  hit.color = hasCol ? unpackUnorm4x8(__float_as_uint(R.v[1].w)) * bary.x + unpackUnorm4x8(__float_as_uint(R.v[2].w)) * bary.y
                           + unpackUnorm4x8(__float_as_uint(R.v[3].w)) * bary.z
                     : f4(1, 1, 1, 1);

  float4 tng0, tng1, tng2;
  if(hasTan)
  {
    tng0 = R.v[9];
    tng1 = R.v[10];
    tng2 = R.v[11];
  }
  else
  {
    tng0 = tng1 = tng2 = makeFastTangent(normal);
  }
  hit.tangent = normalize(xyz(tng0) * bary.x + xyz(tng1) * bary.y + xyz(tng2) * bary.z);
  hit.tangent = xfVector(O2W, hit.tangent);
  hit.tangent = normalize(hit.tangent - hit.nrm * dot(hit.nrm, hit.tangent));
  hit.bitangent = cross(hit.nrm, hit.tangent) * tng0.w;

  if(!frontFace)
    hit.geonrm = -hit.geonrm;
  if(dot(hit.geonrm, hit.nrm) < 0)
  {
    hit.nrm = -hit.nrm;
    hit.tangent = -hit.tangent;
    hit.bitangent = -hit.bitangent;
  }
  const float3 r = reflect(normalize(rayDir), hit.nrm);
  if(dot(r, hit.geonrm) < 0)
    hit.nrm = hit.geonrm;
  return hit;
}

// ---- textures -----------------------------------------------------------------------------------
// 8-bit sRGB EOTF decode table (same fp32 values as the oracle's), staged in shared memory by every kernel
// that can touch a texture (divergent indices: constant memory would serialise them)
extern __shared__ float s_lutSrgb[];
PT_D void stageSrgbLut(const float* __restrict__ lutGlobal)
{
  for(int i = threadIdx.x; i < 512; i += blockDim.x)
    s_lutSrgb[i] = __ldg(lutGlobal + i);
  __syncthreads();
}

// Explicit-LOD fetch.  lambda is computed in fp32 exactly like the Vulkan SampleGrad definition the
// reference relies on: log2(max(|ddx*size|, |ddy*size|)); lambda <= 0 is magnification (level 0).
//
// Filtering is done in fp32 in the kernel from point-sampled texels (bindless texture objects are
// used for the 2D-local fetch path only).  Hardware bilinear/trilinear blends use 8-bit fixed-point
// weights; an alpha-MASK cutoff evaluated on such a blend flips at leaf silhouettes relative to the
// fp32 definition and the paths diverge, so the exact definition is kept (measured: 1e-5 of rays).
// (out of line: the generic modes are rare, and inlining their integer divisions into every texel fetch blew the
// shade kernel up past the instruction cache -- ncu: 42 % of its stall samples were no_instruction)
__device__ __noinline__ int wrapCoord(int i, int n, int mode)
{
  if(mode == 33071)  // CLAMP_TO_EDGE
    return min(max(i, 0), n - 1);
  if(mode == 33648)  // MIRRORED_REPEAT
  {
    const int p = 2 * n;
    const int m = ((i % p) + p) % p;
    return m < n ? m : p - 1 - m;
  }
  return ((i % n) + n) % n;  // REPEAT
}

// texel (x, y) of one level (coordinates already wrapped); `lv` points at the level's first tile, tpr = tiles per row
PT_D float4 fetchTexel(const uchar4* __restrict__ lv, int tpr, bool srgb, int x, int y)
{
  const uchar4 p = __ldg(lv + (((y >> 2) * tpr + (x >> 2)) << 4) + ((y & 3) << 2) + (x & 3));
  const float* lutRgb = srgb ? s_lutSrgb : s_lutSrgb + 256;  // second half: i / 255
  return f4(lutRgb[p.x], lutRgb[p.y], lutRgb[p.z], s_lutSrgb[256 + p.w]);
}

PT_D int wrapFast(int i, int n, int mode)
{
  if(mode == 10497 && (n & (n - 1)) == 0)
    return i & (n - 1);  // REPEAT on a power-of-two level: no integer division
  return wrapCoord(i, n, mode);
}

PT_D float4 sampleLevel(const DevTex& T, int level, float2 uv, bool linear)
{
  const int     w = max(1, T.w0 >> level), h = max(1, T.h0 >> level);
  const uchar4* lv = T.texels + __ldg(T.levelOfs + level);
  const int     tpr = (w + 3) >> 2;
  const bool    srgb = T.srgb != 0;
  float         x = uv.x * (float)w, y = uv.y * (float)h;
  if(!linear)
    return fetchTexel(lv, tpr, srgb, wrapFast((int)floorf(x), w, T.wrapS), wrapFast((int)floorf(y), h, T.wrapT));
  x -= 0.5f;
  y -= 0.5f;
  const float  fx0 = floorf(x), fy0 = floorf(y);
  const float  fx = x - fx0, fy = y - fy0;
  const int    x0 = wrapFast((int)fx0, w, T.wrapS), x1 = wrapFast((int)fx0 + 1, w, T.wrapS);
  const int    y0 = wrapFast((int)fy0, h, T.wrapT), y1 = wrapFast((int)fy0 + 1, h, T.wrapT);
  const float4 a = fetchTexel(lv, tpr, srgb, x0, y0), b = fetchTexel(lv, tpr, srgb, x1, y0);
  const float4 c = fetchTexel(lv, tpr, srgb, x0, y1), d = fetchTexel(lv, tpr, srgb, x1, y1);
  const float4 top = a * (1.0f - fx) + b * fx;
  const float4 bot = c * (1.0f - fx) + d * fx;
  return top * (1.0f - fy) + bot * fy;
}

__device__ __noinline__ float4 sampleTexture(const DevTex& T, float2 uv, float2 ddx, float2 ddy, bool useGrad)
{
  if(!useGrad)
    return sampleLevel(T, 0, uv, T.magLinear != 0);
  const float w = (float)T.w0, h = (float)T.h0;
  const float lx = sqrtf(ddx.x * w * ddx.x * w + ddx.y * h * ddx.y * h);
  const float ly = sqrtf(ddy.x * w * ddy.x * w + ddy.y * h * ddy.y * h);
  float       lambda = log2f(fmaxf(lx, ly));
  if(!(lambda > 0.0f))
    return sampleLevel(T, 0, uv, T.magLinear != 0);
  lambda = fminf(lambda, T.maxLevel);
  if(!T.mipLinear)
  {
    const int lv = (int)fminf(T.maxLevel, fmaxf(0.0f, ceilf(lambda + 0.5f) - 1.0f));
    return sampleLevel(T, lv, uv, T.minLinear != 0);
  }
  const int    l0 = (int)floorf(lambda);
  const int    l1 = min(l0 + 1, (int)T.maxLevel);
  const float  f = lambda - (float)l0;
  const float4 a = sampleLevel(T, l0, uv, T.minLinear != 0);
  if(f == 0.0f || l1 == l0)
    return a;
  const float4 b = sampleLevel(T, l1, uv, T.minLinear != 0);
  return a * (1.0f - f) + b * f;
}

__device__ __noinline__ float4 getTexture(const DevScene& S, uint16_t slot, float2 tc0, float2 tc1, float texGrad)
{
  const b200pt_texture_info ti = S.texInfos[slot];
  float2                    tt = ti.texCoord ? tc1 : tc0;
  const float*              m = ti.uvTransform;
  tt = f2(m[0] * tt.x + m[2] * tt.y + m[4], m[1] * tt.x + m[3] * tt.y + m[5]);
  if(ti.index < 0 || ti.index >= S.numTextures)
    return f4(1, 1, 1, 1);
  const DevTex T = S.textures[ti.index];
  if(texGrad > 0.0f)
    return sampleTexture(T, tt, f2(m[0] * texGrad, m[1] * texGrad), f2(m[2] * texGrad, m[3] * texGrad), true);
  return sampleTexture(T, tt, f2(0, 0), f2(0, 0), false);
}
PT_D float4 sampleLevel0(const DevScene& S, const b200pt_texture_info& ti, float2 uv)
{
  if(ti.index < 0 || ti.index >= S.numTextures)
    return f4(1, 1, 1, 1);
  const DevTex T = S.textures[ti.index];
  return sampleLevel(T, 0, uv, T.magLinear != 0);
}

// ---- material evaluation ------------------------------------------------------------------------
#define PT_MICROFACET_MIN_ROUGHNESS 0.0014142f

PT_D float3 multiToSingleScatterAlbedo(float3 rho)
{
  const float3 t = f3(4.09712f) + rho * 4.20863f - sqrtv(f3(9.59217f) + rho * 41.6808f + rho * rho * 17.7126f);
  return f3(1.0f) - t * t;
}

template <uint32_t FEAT>
PT_D PbrMaterial evaluateMaterial(const DevScene& S, const b200pt_shade_material& material, const HitState& hit, bool isInside, float texGrad)
{
  PbrMaterial pbrMat;
#define PT_TEX(slot) getTexture(S, material.slot, hit.uv0, hit.uv1, texGrad)
  if((FEAT & FEAT_SPECGLOSS) && material.pbrModel == 1)
  {
    // KHR_materials_pbrSpecularGlossiness -> metallic-roughness (gltf_material_eval.h.slang:136-161,176-197)
    float4 diffuse = f4(material.pbrDiffuseFactor[0], material.pbrDiffuseFactor[1], material.pbrDiffuseFactor[2], material.pbrDiffuseFactor[3]) * hit.color;
    float  glossiness = material.pbrGlossinessFactor;
    float3 specular = f3(material.pbrSpecularFactor[0], material.pbrSpecularFactor[1], material.pbrSpecularFactor[2]);
    if(material.pbrDiffuseTexture > 0)
      diffuse *= PT_TEX(pbrDiffuseTexture);
    if(material.pbrSpecularGlossinessTexture > 0)
    {
      const float4 s = PT_TEX(pbrSpecularGlossinessTexture);
      specular *= xyz(s);
      glossiness *= s.w;
    }
    const float ds = 0.04f;
    const float specI = fmaxf(specular.x, fmaxf(specular.y, specular.z));
    pbrMat.metallic = smoothstepf(ds + 0.01f, ds + 0.05f, specI);
    if(pbrMat.metallic > 0.0f)
      pbrMat.baseColor = specular;
    else
    {
      float3 bc = xyz(diffuse) / (1.0f - ds * (1.0f - pbrMat.metallic));
      pbrMat.baseColor = f3(clampf(bc.x, 0, 1), clampf(bc.y, 0, 1), clampf(bc.z, 0, 1));
    }
    const float r = 1.0f - glossiness;
    pbrMat.roughness = f2(r * r, r * r);
    pbrMat.opacity = diffuse.w;
  }
  else
  {
    float4 baseColor = f4(material.pbrBaseColorFactor[0], material.pbrBaseColorFactor[1], material.pbrBaseColorFactor[2], material.pbrBaseColorFactor[3]) * hit.color;
    if(material.pbrBaseColorTexture > 0)
      baseColor *= PT_TEX(pbrBaseColorTexture);
    pbrMat.baseColor = xyz(baseColor);
    pbrMat.opacity = baseColor.w;
    float roughness = material.pbrRoughnessFactor;
    float metallic = material.pbrMetallicFactor;
    if(material.pbrMetallicRoughnessTexture > 0)
    {
      const float4 mr = PT_TEX(pbrMetallicRoughnessTexture);
      roughness *= mr.y;
      metallic *= mr.z;
    }
    roughness = fmaxf(roughness, PT_MICROFACET_MIN_ROUGHNESS);
    pbrMat.roughness = f2(roughness * roughness, roughness * roughness);
    pbrMat.metallic = clampf(metallic, 0.0f, 1.0f);
  }
  // occlusion (gltf_material_eval.h.slang:228-233) is fetched by the reference but never read by the path tracer
  // (only the rasteriser's ambient term uses it): not evaluated here, no effect on the image

  pbrMat.N = hit.nrm;
  pbrMat.T = hit.tangent;
  pbrMat.B = hit.bitangent;
  pbrMat.Ng = hit.geonrm;
  bool needsTangentUpdate = false;
  if(material.normalTexture > 0)
  {
    float3 nv = xyz(PT_TEX(normalTexture));
    nv = nv * 2.0f - f3(1.0f);
    nv = nv * f3(material.normalTextureScale, material.normalTextureScale, 1.0f);
    pbrMat.N = normalize(hit.tangent * nv.x + hit.bitangent * nv.y + hit.nrm * nv.z);
    needsTangentUpdate = true;
  }

  pbrMat.emissive = f3(material.emissiveFactor[0], material.emissiveFactor[1], material.emissiveFactor[2]);
  if(material.emissiveTexture > 0)
    pbrMat.emissive *= xyz(PT_TEX(emissiveTexture));
  pbrMat.emissive = vmax(f3(0.0f), pbrMat.emissive);

  pbrMat.attenuationColor = f3(material.attenuationColor[0], material.attenuationColor[1], material.attenuationColor[2]);
  pbrMat.attenuationDistance = material.attenuationDistance;
  pbrMat.thickness = material.thicknessFactor;
  if((FEAT & FEAT_VOLUME) && material.thicknessTexture > 0)
    pbrMat.thickness *= PT_TEX(thicknessTexture).y;

  pbrMat.specularColor = f3(material.specularColorFactor[0], material.specularColorFactor[1], material.specularColorFactor[2]);
  if(material.specularColorTexture > 0)
    pbrMat.specularColor *= xyz(PT_TEX(specularColorTexture));
  pbrMat.specular = material.specularFactor;
  if(material.specularTexture > 0)
    pbrMat.specular *= PT_TEX(specularTexture).w;

  float ior1 = 1.0f, ior2 = material.ior;
  if(isInside && (pbrMat.thickness > 0.0f))
  {
    ior1 = ior2;
    ior2 = 1.0f;
  }
  pbrMat.ior1 = ior1;
  pbrMat.ior2 = ior2;

  pbrMat.transmission = material.transmissionFactor;
  if((FEAT & FEAT_TRANSMISSION) && material.transmissionTexture > 0)
    pbrMat.transmission *= PT_TEX(transmissionTexture).x;

  pbrMat.scatterCoefficient = f3(0.0f);
  if((FEAT & FEAT_VOLUME) && (material.multiscatterColorFactor[0] > 0.0f || material.multiscatterColorFactor[1] > 0.0f || material.multiscatterColorFactor[2] > 0.0f))
  {
    const float3 ssa = multiToSingleScatterAlbedo(f3(material.multiscatterColorFactor[0], material.multiscatterColorFactor[1], material.multiscatterColorFactor[2]));
    const float3 att = -logv(vmax(pbrMat.attenuationColor, f3(0.001f))) / fmaxf(pbrMat.attenuationDistance, 0.001f);
    pbrMat.scatterCoefficient = att * ssa;
  }
  pbrMat.scatterAnisotropy = material.scatterAnisotropy;

  pbrMat.clearcoat = material.clearcoatFactor;
  pbrMat.clearcoatRoughness = material.clearcoatRoughness;
  pbrMat.Nc = pbrMat.N;
  if((FEAT & FEAT_CLEARCOAT) && material.clearcoatTexture > 0)
    pbrMat.clearcoat *= PT_TEX(clearcoatTexture).x;
  if((FEAT & FEAT_CLEARCOAT) && material.clearcoatRoughnessTexture > 0)
    pbrMat.clearcoatRoughness *= PT_TEX(clearcoatRoughnessTexture).y;
  if((FEAT & FEAT_CLEARCOAT) && material.clearcoatNormalTexture > 0)
  {
    float3 nv = xyz(PT_TEX(clearcoatNormalTexture));
    nv = nv * 2.0f - f3(1.0f);
    pbrMat.Nc = normalize(pbrMat.T * nv.x + pbrMat.B * nv.y + pbrMat.Nc * nv.z);
  }
  pbrMat.clearcoatRoughness = fmaxf(pbrMat.clearcoatRoughness, 0.001f);

  float iridescence = material.iridescenceFactor;
  float iridescenceThickness = material.iridescenceThicknessMaximum;
  pbrMat.iridescenceIor = material.iridescenceIor;
  if((FEAT & FEAT_IRIDESCENCE) && material.iridescenceTexture > 0)
    iridescence *= PT_TEX(iridescenceTexture).x;
  if((FEAT & FEAT_IRIDESCENCE) && material.iridescenceThicknessTexture > 0)
  {
    const float t = PT_TEX(iridescenceThicknessTexture).y;
    iridescenceThickness = lerpf(material.iridescenceThicknessMinimum, material.iridescenceThicknessMaximum, t);
  }
  pbrMat.iridescence = (iridescenceThickness > 0.0f) ? iridescence : 0.0f;
  pbrMat.iridescenceThickness = iridescenceThickness;

  float anisotropyStrength = material.anisotropyStrength;
  if((FEAT & FEAT_ANISOTROPY) && anisotropyStrength > 0.0f)
  {
    float2 dir = f2(1.0f, 0.0f);
    if(material.anisotropyTexture > 0)
    {
      const float4 at = PT_TEX(anisotropyTexture);
      dir = normalize(f2(at.x * 2.0f - 1.0f, at.y * 2.0f - 1.0f));
      anisotropyStrength *= at.z;
    }
    pbrMat.roughness.x = lerpf(pbrMat.roughness.y, 1.0f, anisotropyStrength * anisotropyStrength);
    const float s = material.anisotropyRotation[0], c = material.anisotropyRotation[1];
    dir = f2(c * dir.x + s * dir.y, c * dir.y - s * dir.x);
    pbrMat.T = pbrMat.T * dir.x + pbrMat.B * dir.y;
    needsTangentUpdate = true;
  }

  if(needsTangentUpdate)
  {
    pbrMat.B = normalize(cross(pbrMat.N, pbrMat.T));
    const float bitangentSign = signf(dot(hit.bitangent, pbrMat.B));
    pbrMat.B = pbrMat.B * bitangentSign;
    pbrMat.T = normalize(cross(pbrMat.B, pbrMat.N) * bitangentSign);
  }

  pbrMat.sheenColor = f3(material.sheenColorFactor[0], material.sheenColorFactor[1], material.sheenColorFactor[2]);
  if((FEAT & FEAT_SHEEN) && material.sheenColorTexture > 0)
    pbrMat.sheenColor *= xyz(PT_TEX(sheenColorTexture));
  pbrMat.sheenRoughness = material.sheenRoughnessFactor;
  if((FEAT & FEAT_SHEEN) && material.sheenRoughnessTexture > 0)
    pbrMat.sheenRoughness *= PT_TEX(sheenRoughnessTexture).w;
  pbrMat.sheenRoughness = fmaxf(PT_MICROFACET_MIN_ROUGHNESS, pbrMat.sheenRoughness);

  pbrMat.diffuseTransmissionFactor = material.diffuseTransmissionFactor;
  if((FEAT & FEAT_DIFFUSE_TRANSMISSION) && material.diffuseTransmissionTexture > 0)
    pbrMat.diffuseTransmissionFactor *= PT_TEX(diffuseTransmissionTexture).w;
  pbrMat.diffuseTransmissionColor = f3(material.diffuseTransmissionColor[0], material.diffuseTransmissionColor[1], material.diffuseTransmissionColor[2]);
  if((FEAT & FEAT_DIFFUSE_TRANSMISSION) && material.diffuseTransmissionColorTexture > 0)
    pbrMat.diffuseTransmissionColor *= xyz(PT_TEX(diffuseTransmissionColorTexture));
  // KHR_materials_dispersion (gltf_material_eval.h.slang:426-428); evaluated on the specular-transmission lobe (bsdf.cuh)
  pbrMat.dispersion = (FEAT & FEAT_TRANSMISSION) ? material.dispersion : 0.0f;
  // KHR_materials_retroreflection (:447-452): the lobe itself lives in nvshaders (external, not restated): scenes that
  // use it are rejected by b200pt_set_scene, so the factor is always 0 here
  pbrMat.retroreflection = 0.0f;
#undef PT_TEX
  return pbrMat;
}

// ---- alpha + shadow transmission ----------------------------------------------------------------
PT_D float getOpacity(const DevScene& S, const b200pt_render_node& node, const DevPrim& P, uint32_t triangleID, float3 bary)
{
  const b200pt_shade_material& mat = S.mats[max(0, node.materialID)];
  if(mat.alphaMode == 0)
    return 1.0f;
  const uint3 tri = loadTri(P, triangleID);
  float       a;
  if(mat.pbrModel == 1)
  {
    a = mat.pbrDiffuseFactor[3];
    if(mat.pbrDiffuseTexture > 0)
    {
      const b200pt_texture_info ti = S.texInfos[mat.pbrDiffuseTexture];
      a *= sampleLevel0(S, ti, interpTexCoord(P, ti.texCoord, tri, bary)).w;
    }
  }
  else
  {
    a = mat.pbrBaseColorFactor[3];
    if(mat.pbrBaseColorTexture > 0)
    {
      const b200pt_texture_info ti = S.texInfos[mat.pbrBaseColorTexture];
      a *= sampleLevel0(S, ti, interpTexCoord(P, ti.texCoord, tri, bary)).w;
    }
  }
  a *= interpColor(P, tri, bary).w;
  if(mat.alphaMode == 1)
    return a >= mat.alphaCutoff ? 1.0f : 0.0f;
  return a;
}

PT_D AlphaRec loadAlphaRec(const AlphaRec* __restrict__ p)
{
  // four 128-bit loads
  const float4* q = reinterpret_cast<const float4*>(p);
  union
  {
    float4   v[4];
    AlphaRec r;
  } u;
  u.v[0] = __ldg(q + 0);
  u.v[1] = __ldg(q + 1);
  u.v[2] = __ldg(q + 2);
  u.v[3] = __ldg(q + 3);
  return u.r;
}

// getOpacity from the pre-gathered record: the same arithmetic, operation by operation, as the generic function above
// (interpolated uv, level-0 fetch with the magnification filter, vertex-colour alpha, MASK cutoff)
PT_D float opacityFromRecord(const AlphaRec& r, float3 bary)
{
  const uint32_t mode = r.modeFlags & 3u;
  if(mode == 0u)
    return 1.0f;
  float a = r.factor;
  if(r.lv0 != nullptr)
  {
    const float2 uv = f2(r.uv[0], r.uv[1]) * bary.x + f2(r.uv[2], r.uv[3]) * bary.y + f2(r.uv[4], r.uv[5]) * bary.z;
    const int    w = r.w0, h = r.h0, tpr = (w + 3) >> 2;
    const int    wrapS = (int)(r.wrap & 0xffffu), wrapT = (int)(r.wrap >> 16);
    float        x = uv.x * (float)w, y = uv.y * (float)h;
    auto         alphaAt = [&](int tx, int ty) { return s_lutSrgb[256 + __ldg(r.lv0 + (((ty >> 2) * tpr + (tx >> 2)) << 4) + ((ty & 3) << 2) + (tx & 3)).w]; };
    if(!(r.modeFlags & 4u))
      a *= alphaAt(wrapFast((int)floorf(x), w, wrapS), wrapFast((int)floorf(y), h, wrapT));
    else
    {
      x -= 0.5f;
      y -= 0.5f;
      const float fx0 = floorf(x), fy0 = floorf(y);
      const float fx = x - fx0, fy = y - fy0;
      const int   x0 = wrapFast((int)fx0, w, wrapS), x1 = wrapFast((int)fx0 + 1, w, wrapS);
      const int   y0 = wrapFast((int)fy0, h, wrapT), y1 = wrapFast((int)fy0 + 1, h, wrapT);
      const float ta = alphaAt(x0, y0), tb = alphaAt(x1, y0), tc = alphaAt(x0, y1), td = alphaAt(x1, y1);
      const float top = ta * (1.0f - fx) + tb * fx;
      const float bot = tc * (1.0f - fx) + td * fx;
      a *= top * (1.0f - fy) + bot * fy;
    }
  }
  if(r.modeFlags & 8u)
  {
    const float a0 = (float)(r.colA & 0xffu) / 255.0f, a1 = (float)((r.colA >> 8) & 0xffu) / 255.0f, a2 = (float)((r.colA >> 16) & 0xffu) / 255.0f;
    a *= a0 * bary.x + a1 * bary.y + a2 * bary.z;
  }
  if(mode == 1u)
    return a >= r.cutoff ? 1.0f : 0.0f;
  return a;
}

PT_D float3 getShadowTransmission(const DevScene& S, const b200pt_render_node& node, const DevPrim& P, uint32_t triangleID, float3 bary, float hitT, float3 rayDir, bool& isInside)
{
  const b200pt_shade_material& mat = S.mats[max(0, node.materialID)];
  const float                  tFactor = mat.transmissionFactor;
  if(tFactor <= 0.01f)
    return f3(0.0f);
  const uint3 tri = loadTri(P, triangleID);
  float3      normal;
  {
    const float3 v0 = ld3(P.pos, tri.x), v1 = ld3(P.pos, tri.y), v2 = ld3(P.pos, tri.z);
    normal = normalize(cross(v1 - v0, v2 - v0));
    normal = normalize(xfNormal(node.worldToObject, normal));
  }
  const float cosTheta = fabsf(dot(rayDir, normal));
  const float fresnel = schlickFresnel(mat.ior, cosTheta);
  float3      cur = f3(mat.pbrBaseColorFactor[0], mat.pbrBaseColorFactor[1], mat.pbrBaseColorFactor[2]) * tFactor;
  cur *= (1.0f - fresnel);
  if(mat.thicknessFactor > 0.0f)
  {
    if(isInside)
    {
      const float3 absCoeff = -logv(vmax(f3(mat.attenuationColor[0], mat.attenuationColor[1], mat.attenuationColor[2]), f3(0.001f))) / fmaxf(mat.attenuationDistance, 0.001f);
      const float3 scatterCoeff = absCoeff * multiToSingleScatterAlbedo(f3(mat.multiscatterColorFactor[0], mat.multiscatterColorFactor[1], mat.multiscatterColorFactor[2]));
      const float3 extinction = absCoeff + scatterCoeff;
      cur *= expv(extinction * -hitT);
      if(maxc(scatterCoeff) > 0.001f)
        cur *= expf(-(hitT * maxc(extinction)));
    }
    isInside = !isInside;
  }
  float att = 1.0f;
  {
    float roughness = mat.pbrRoughnessFactor, metallic = mat.pbrMetallicFactor;
    if(mat.pbrMetallicRoughnessTexture > 0)
    {
      const b200pt_texture_info ti = S.texInfos[mat.pbrMetallicRoughnessTexture];
      const float4              mr = sampleLevel0(S, ti, interpTexCoord(P, ti.texCoord, tri, bary));
      roughness *= mr.y;
      metallic *= mr.z;
    }
    att *= (1.0f - metallic);
    const float roughnessEffect = 1.0f - (roughness * roughness);
    att *= lerpf(0.65f, 1.0f, roughnessEffect);
  }
  return cur * att;
}

// ---- Trace / TraceShadow -------------------------------------------------------------------------
// The reference leaves any-hit order to the hardware (raytracer_interface.h.slang:53).  Pinned here:
//   Trace:       closest FORCE_OPAQUE hit, then the non-opaque candidates nearer than it front-to-back in
//                (t, triangle id) order, one rand() each.
//   TraceShadow: any opaque occluder => 0 with no rand(); else every non-opaque candidate front-to-back.
// Geometry: traverse.cuh (one walk per ray: k_trace / k_shadow); alpha tests + transmission: k_alpha (b200pt.cu).

// ---- environment --------------------------------------------------------------------------------
// lat-long lookup with fp32 bilinear weights (linear filter, level 0, repeat in u / clamp in v)
PT_D float4 sampleEnvTex(const DevScene& S, float2 uv)
{
  const int   w = S.envW, h = S.envH;
  const float x = uv.x * (float)w - 0.5f, y = uv.y * (float)h - 0.5f;
  const float fx0 = floorf(x), fy0 = floorf(y);
  const float fx = x - fx0, fy = y - fy0;
  int         x0 = (int)fx0, y0 = (int)fy0;
  int         x1 = x0 + 1, y1 = y0 + 1;
  x0 = ((x0 % w) + w) % w;
  x1 = ((x1 % w) + w) % w;
  y0 = min(max(y0, 0), h - 1);
  y1 = min(max(y1, 0), h - 1);
  const float4 a = __ldg(&S.envRgba[(size_t)y0 * w + x0]), b = __ldg(&S.envRgba[(size_t)y0 * w + x1]);
  const float4 c = __ldg(&S.envRgba[(size_t)y1 * w + x0]), d = __ldg(&S.envRgba[(size_t)y1 * w + x1]);
  const float4 top = a * (1.0f - fx) + b * fx;
  const float4 bot = c * (1.0f - fx) + d * fx;
  return top * (1.0f - fy) + bot * fy;
}

PT_D float4 environmentSample(const DevScene& S, float3 xi, float3& toLight)
{
  const uint32_t width = (uint32_t)S.envW, height = (uint32_t)S.envH;
  const uint32_t size = width * height;
  const uint32_t idx = min((uint32_t)(xi.x * (float)size), size - 1);
  const uint2    acc = __ldg(&S.envAccel[idx]);
  const float    q = __uint_as_float(acc.y);
  uint32_t       envIdx;
  float          xi_y = xi.y;
  if(xi_y < q)
  {
    envIdx = idx;
    xi_y /= q;
  }
  else
  {
    envIdx = acc.x;
    xi_y = (xi_y - q) / (1.0f - q);
  }
  const uint32_t py = envIdx / width;
  const uint32_t px = envIdx % width;
  const float    u = ((float)px + xi_y) / (float)width;
  const float    phi = u * kTwoPi - kPi;
  const float    sinPhi = sinf(phi), cosPhi = cosf(phi);
  const float    stepTheta = kPi / (float)height;
  const float    theta0 = (float)py * stepTheta;
  const float    cosTheta = cosf(theta0) * (1.0f - xi.z) + cosf(theta0 + stepTheta) * xi.z;
  const float    theta = acosf(cosTheta);
  const float    sinTheta = sinf(theta);
  const float    v = theta * kInvPi;
  toLight = f3(cosPhi * sinTheta, cosTheta, sinPhi * sinTheta);
  return sampleEnvTex(S, f2(u, v));
}

// ---- punctual lights ----------------------------------------------------------------------------
struct LightContrib
{
  float3 incidentVector;
  float3 intensity;
  float  distance;
  float  pdf;
};

PT_D LightContrib singleLightContribution(const b200pt_light& light, float3 surfacePos, float2 xi)
{
  LightContrib c;
  c.incidentVector = f3(0.0f);
  c.intensity = f3(0.0f);
  c.distance = kInfinite;
  c.pdf = kDirac;
  float        halfAngularSize = 0.0f;
  float        irradiance = 0.0f;
  const float3 ldir = f3(light.direction[0], light.direction[1], light.direction[2]);
  if(light.type == 1)
  {
    c.incidentVector = ldir;
    halfAngularSize = light.angularSizeOrInvRange * 0.5f;
    irradiance = light.intensity;
  }
  else if(light.type == 2 || light.type == 3)
  {
    const float3 l2s = surfacePos - f3(light.position[0], light.position[1], light.position[2]);
    const float  distance = sqrtf(dot(l2s, l2s));
    const float  rDistance = 1.0f / distance;
    c.distance = distance;
    c.incidentVector = l2s * rDistance;
    float attenuation = 1.0f;
    if(light.angularSizeOrInvRange > 0.0f)
    {
      attenuation = square(saturatef(1.0f - square(square(distance * light.angularSizeOrInvRange))));
      if(attenuation == 0.0f)
        return c;
    }
    float spotlight = 1.0f;
    if(light.type == 2)
    {
      const float lDotD = dot(c.incidentVector, ldir);
      const float directionAngle = acosf(clampf(lDotD, -1.0f, 1.0f));
      spotlight = 1.0f - smoothstepf(light.innerAngle, light.outerAngle, directionAngle);
      if(spotlight == 0.0f)
        return c;
    }
    if(light.radius > 0.0f)
    {
      halfAngularSize = atanf(fminf(light.radius * rDistance, 1.0f));
      const float solidAngleOverPi = square(halfAngularSize);
      const float radianceTimesPi = light.intensity / square(light.radius);
      irradiance = radianceTimesPi * solidAngleOverPi;
    }
    else
      irradiance = light.intensity * square(rDistance);
    irradiance *= spotlight * attenuation;
  }
  c.intensity = f3(light.color[0], light.color[1], light.color[2]) * irradiance;
  if(halfAngularSize > 0.0f)
  {
    const float  cosMax = cosf(halfAngularSize);
    const float  cosT = 1.0f - xi.x * (1.0f - cosMax);
    const float  sinT = sqrtf(fmaxf(0.0f, 1.0f - cosT * cosT));
    const float  phi = kTwoPi * xi.y;
    const float3 axis = -c.incidentVector;
    const float3 T = normalize(xyz(makeFastTangent(axis)));
    const float3 B = cross(axis, T);
    const float3 d = normalize(T * (sinT * cosf(phi)) + B * (sinT * sinf(phi)) + axis * cosT);
    c.incidentVector = -d;
    c.pdf = 1.0f / (kTwoPi * (1.0f - cosMax));
  }
  return c;
}

struct DirectLight
{
  float3 direction, radianceOverPdf;
  float  distance, pdf;
};

PT_D void techniqueProbabilities(const DevScene& S, const FrameParams& F, float& lightWeight, float& envWeight)
{
  lightWeight = (S.numLights > 0) ? 0.5f : 0.0f;
  envWeight = (!(F.fi.flags & B200PT_SCENE_USE_HDR_ENVIRONMENT) || F.fi.envIntensity > 0.0f) ? 0.5f : 0.0f;
  const float total = lightWeight + envWeight;
  if(total > 0.0f)
  {
    lightWeight /= total;
    envWeight /= total;
  }
}

template <uint32_t FEAT>
PT_D DirectLight sampleLights(const DevScene& S, const FrameParams& F, float3 pos, uint32_t& seed)
{
  DirectLight dl;
  float3      radiance = f3(0.0f);
  dl.pdf = 0.0f;
  dl.distance = kInfinite;
  dl.radianceOverPdf = f3(0.0f);
  dl.direction = f3(0.0f);
  float envPdf = 0.0f;
  float lightWeight, envWeight;
  techniqueProbabilities(S, F, lightWeight, envWeight);
  if(lightWeight == 0.0f && envWeight == 0.0f)
    return dl;
  const bool sampleLight = (rnd(seed) < lightWeight);
  if((FEAT & FEAT_LIGHTS) && sampleLight)
  {
    const float         selectionPdf = 1.0f / (float)S.numLights;
    const int           lightIndex = min((int)(rnd(seed) * (float)S.numLights), S.numLights - 1);
    const b200pt_light& light = S.lights[lightIndex];
    const float         r1 = rnd(seed), r2 = rnd(seed);
    const LightContrib  contrib = singleLightContribution(light, pos, f2(r1, r2));
    dl.direction = -contrib.incidentVector;
    dl.distance = contrib.distance;
    radiance = contrib.intensity / (selectionPdf * lightWeight);
    dl.pdf = (contrib.pdf == kDirac) ? kDirac : selectionPdf * contrib.pdf;
  }
  if(envWeight > 0 && dl.pdf != kDirac)
  {
    if(!sampleLight)
    {
      const float  a = rnd(seed), b = rnd(seed), c = rnd(seed);
      const float4 rp = environmentSample(S, f3(a, b, c), dl.direction);
      envPdf = rp.w;
      radiance = xyz(rp) * F.fi.envIntensity / (envPdf * envWeight);
      dl.direction = rotateAxis(dl.direction, f3(0, 1, 0), F.fi.envRotation);
    }
    else
    {
      const float3 dir = rotateAxis(dl.direction, f3(0, 1, 0), -F.fi.envRotation);
      envPdf = sampleEnvTex(S, getSphericalUv(dir)).w;
    }
  }
  float misWeight = 1.0f;
  if(dl.pdf != kDirac)
  {
    const float pdfSum = lightWeight * dl.pdf + envWeight * envPdf;
    if(pdfSum > 0.0f)
      misWeight = (sampleLight ? lightWeight * dl.pdf : envWeight * envPdf) / pdfSum;
    dl.pdf = pdfSum;
  }
  radiance *= misWeight;
  dl.radianceOverPdf = radiance;
  return dl;
}

// ---- volume medium (fp16 storage like the reference's float16_t fields) --------------------------
struct VolumeMedium
{
  float3 extinction, scatterCoefficient;
  float  scatterAnisotropy;
};
PT_D float  roundHalf(float f) { return __half2float(__float2half_rn(f)); }
PT_D uint4 packMedium(const VolumeMedium& m, uint32_t w)
{
  uint4 p;
  p.x = (uint32_t)__half_as_ushort(__float2half_rn(m.extinction.x)) | ((uint32_t)__half_as_ushort(__float2half_rn(m.extinction.y)) << 16);
  p.y = (uint32_t)__half_as_ushort(__float2half_rn(m.extinction.z)) | ((uint32_t)__half_as_ushort(__float2half_rn(m.scatterCoefficient.x)) << 16);
  p.z = (uint32_t)__half_as_ushort(__float2half_rn(m.scatterCoefficient.y)) | ((uint32_t)__half_as_ushort(__float2half_rn(m.scatterCoefficient.z)) << 16);
  p.w = (uint32_t)__half_as_ushort(__float2half_rn(m.scatterAnisotropy)) | (w << 16);
  return p;
}
PT_D VolumeMedium unpackMedium(uint4 p)
{
  VolumeMedium m;
  m.extinction = f3(__half2float(__ushort_as_half(p.x & 0xffff)), __half2float(__ushort_as_half(p.x >> 16)), __half2float(__ushort_as_half(p.y & 0xffff)));
  m.scatterCoefficient = f3(__half2float(__ushort_as_half(p.y >> 16)), __half2float(__ushort_as_half(p.z & 0xffff)), __half2float(__ushort_as_half(p.z >> 16)));
  m.scatterAnisotropy = __half2float(__ushort_as_half(p.w & 0xffff));
  return m;
}
PT_D VolumeMedium makeVolumeMedium(const PbrMaterial& m)
{
  VolumeMedium v;
  const float3 absC = -logv(vmax(m.attenuationColor, f3(0.001f))) / fmaxf(m.attenuationDistance, 0.001f);
  v.extinction = absC + m.scatterCoefficient;
  v.scatterCoefficient = m.scatterCoefficient;
  v.scatterAnisotropy = m.scatterAnisotropy;
  return v;
}
PT_D bool hasVolumeMedium(const VolumeMedium& v) { return maxc(v.extinction) > 0.0f || maxc(v.scatterCoefficient) > 0.0f; }

}  // namespace pt
