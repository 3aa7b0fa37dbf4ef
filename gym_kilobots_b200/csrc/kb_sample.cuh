// kb_sample.cuh -- random scene initialisation at reset, on the device, inside the reset kernel.
//
// Restates what YamlKilobotsEnv._configure_environment draws for ONE env with numpy's global generator
// (gym_kilobots/envs/yaml_kilobots_env.py:194-198 objects, :256-283 lights, :299 shuffle of the composite light's
// components, :327-354 kilobots) as a pure function of (seed, GLOBAL env id, episode count): every draw is one
// Philox4x32-10 block keyed by the seed with counter (draw index, stream + 256 * episode, env id), so a reset does
// not depend on the batch size, on the rank count or on which other envs are reset in the same launch.
// gym_kilobots_b200/sampler.py evaluates the same function in numpy (tests compare the two).
//
//   objects   mode RANDOM: position = (U^2 * size + lo) * 0.7, orientation = U * 2 pi - pi; FIXED: the given pose
//   shuffle   Fisher-Yates over the composite light's components; every permutation is a scene template of the batch
//             (light constants are held per scene), the env's scene index is switched at reset
//   lights    RANDOM: U^2 * size + lo; AT_OBJECT: on a circle of radius 1.2 * max(w, h) / 2 around a uniformly chosen
//             object; FIXED; momentum lights start with speed .01 in a uniform direction; linear: the given angle
//   kilobots  mean = the light (one positional light), a uniformly chosen positional light per kilobot (several),
//             U^2 * size + lo scaled by 0.9 (RANDOM), or FIXED; position = mean + std * N(0, 1)^2 clipped to the
//             table -+ 0.02; orientation 0
//
// A batch may mix K configurations (kb_set_sampler_mix): one SamplerConst each.  The reset first picks the env's
// configuration -- drawn from the cumulative weights (stream KS_CONFIG) or looked up from the env's scene -- and then
// draws that configuration's scene as above, in the batch's padded body layout (objects at 0..M_e-1, kilobots at
// Mmax + k; the rows of absent bodies are quiet NaN).
#pragma once
#include "kb_types.cuh"

namespace kb {

#define KB_SAMPLE_MAX_OBJECTS 16
// streams: must match gym_kilobots_b200/philox.py
#define KS_LIGHT 1
#define KS_OBJECT 2
#define KS_KILOBOT_POS 3
#define KS_SWARM 5
#define KS_SHUFFLE 6
#define KS_CONFIG 8
#define KS_ACTUATION 9         // per-episode actuation draws (kb_env.cuh)
#define KS_ACTUATION_NOISE 10  // per-sub-step actuation noise (kb_env.cuh)

struct SamplerConst {
  uint32_t seedLo, seedHi;
  int64_t envIdBase;
  double sizeX, sizeY;                 // table size (m); the table is centred at the origin
  int32_t numObjects, numLights, shuffle, meanMode;   // meanMode: 0 fixed, 1 light, 2 random
  double mean[2], std;
  int32_t objMode[KB_SAMPLE_MAX_OBJECTS];             // 0 fixed, 1 random
  double objPose[KB_SAMPLE_MAX_OBJECTS][3];
  double objExtent[KB_SAMPLE_MAX_OBJECTS];            // max(width, height) as the light placement reads it
  int32_t lightMode[KB_MAX_LIGHTS];                   // per CANONICAL component: 0 fixed, 1 random, 2 at object
  double lightInit[KB_MAX_LIGHTS][2];
  int32_t permScene[24];                              // scene index of every permutation (lexicographic rank)
  int32_t ownScene;                                   // 1: the reset moves the env to permScene[0] (no shuffle, K > 1)
};

struct Philox4 {
  uint32_t x, y, z, w;
};
__device__ __forceinline__ Philox4 philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
  return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) / 9007199254740992.0;
}

struct EnvRng {
  uint32_t k0, k1, e0, e1, ep;
  __device__ __forceinline__ void uniform2(uint32_t stream, uint32_t index, double* u0, double* u1) const {
    const Philox4 r = philox4x32(index, stream + (ep << 8), e0, e1, k0, k1);
    *u0 = u53(r.x, r.y);
    *u1 = u53(r.z, r.w);
  }
  __device__ __forceinline__ void normal2(uint32_t stream, uint32_t index, double* z0, double* z1) const {
    double u0, u1;
    uniform2(stream, index, &u0, &u1);
    const double r = sqrt(-2.0 * log(1.0 - u0));
    const double a = 6.283185307179586 * u1;
    *z0 = r * cos(a);
    *z1 = r * sin(a);
  }
};

// Draws the scene of one env.  lane / nlanes: the threads that cooperate on this env; sync(): their barrier (global
// writes of the group are visible to the group after it).  The draws go to the env's rows of the handle's sample
// buffers (a.samplePose [B][3], a.sampleLight [L]).  KA is KernelArgs (kb_step.cuh): a.sampler[a.numConfigs] are the
// configurations, a.configCdf their cumulative weights (null: a.sceneConfig[sceneIn] is the env's configuration).
// Returns the env's scene index.
template <class KA, class SyncFn>
__device__ __forceinline__ int sampleScene(const KA& a, int env, int sceneIn, uint32_t episode, int lane, int nlanes,
                                           SyncFn sync) {
  const long long envGlobal = a.sampler->envIdBase + env;
  const int B = a.L.B, Mmax = a.L.M;
  double* pose = a.samplePose + (size_t)env * B * 3;
  double* light = a.sampleLight + (size_t)env * (a.L.L > 0 ? a.L.L : 1);
  EnvRng g;
  g.k0 = a.sampler->seedLo;   // seed and env id base agree over the configurations
  g.k1 = a.sampler->seedHi;
  g.e0 = (uint32_t)((unsigned long long)envGlobal & 0xFFFFFFFFull);
  g.e1 = (uint32_t)((unsigned long long)envGlobal >> 32);
  g.ep = episode;
  // ---- configuration (every lane computes the same one)
  int cfg = 0;
  if (a.configCdf) {
    double u, u1;
    g.uniform2(KS_CONFIG, 0u, &u, &u1);
    while (cfg < a.numConfigs - 1 && !(u < a.configCdf[cfg])) ++cfg;
  } else if (a.numConfigs > 1) {
    cfg = max(__ldg(&a.sceneConfig[sceneIn]), 0);
  }
  const SamplerConst* __restrict__ sp = a.sampler + cfg;
  const double pi = 3.141592653589793;
  const double lox = -sp->sizeX / 2, loy = -sp->sizeY / 2;
  const int NL = sp->numLights;
  // ---- composite shuffle (every lane computes the same permutation) -> scene
  int order[KB_MAX_LIGHTS];
#pragma unroll
  for (int i = 0; i < KB_MAX_LIGHTS; ++i) order[i] = i;
  int scene = sceneIn;
  if (sp->shuffle && NL > 1) {
    for (int j = NL - 1; j >= 1; --j) {
      double u0, u1;
      g.uniform2(KS_SHUFFLE, (uint32_t)j, &u0, &u1);
      int r = (int)(u0 * (double)(j + 1));
      r = r > j ? j : r;
      int oj = 0, orr = 0;
#pragma unroll
      for (int i = 0; i < KB_MAX_LIGHTS; ++i) {
        if (i == j) oj = order[i];
        if (i == r) orr = order[i];
      }
#pragma unroll
      for (int i = 0; i < KB_MAX_LIGHTS; ++i) {
        if (i == j) order[i] = orr;
        else if (i == r) order[i] = oj;
      }
    }
    // lexicographic rank of the permutation
    int rank = 0;
    for (int i = 0; i < NL; ++i) {
      int smaller = 0;
      for (int k = i + 1; k < NL; ++k) {
        int oi = 0, ok = 0;
#pragma unroll
        for (int q = 0; q < KB_MAX_LIGHTS; ++q) {
          if (q == i) oi = order[q];
          if (q == k) ok = order[q];
        }
        smaller += ok < oi ? 1 : 0;
      }
      int f = 1;
      for (int q = 2; q <= NL - 1 - i; ++q) f *= q;
      rank += smaller * f;
    }
    scene = sp->permScene[rank];
  } else if (sp->ownScene) {
    scene = sp->permScene[0];
  }
  // ---- this scene's counts; rows of absent bodies are NaN
  const int M = __ldg(&a.scenes[scene].numObjects), N = __ldg(&a.scenes[scene].numKilobots);
  const double qnan = __longlong_as_double(0x7FF8000000000000ll);
  for (int i = lane; i < B; i += nlanes)
    if ((i >= M && i < Mmax) || i >= Mmax + N) pose[3 * i] = pose[3 * i + 1] = pose[3 * i + 2] = qnan;
  // ---- objects
  for (int i = lane; i < M; i += nlanes) {
    double* p = pose + 3 * i;
    if (sp->objMode[i] == 1) {
      double u0, u1, a0, a1;
      g.uniform2(KS_OBJECT, 2u * (uint32_t)i, &u0, &u1);
      g.uniform2(KS_OBJECT, 2u * (uint32_t)i + 1u, &a0, &a1);
      p[0] = (u0 * sp->sizeX + lox) * 0.7;
      p[1] = (u1 * sp->sizeY + loy) * 0.7;
      p[2] = a0 * 2 * pi - pi;
    } else {
      p[0] = sp->objPose[i][0];
      p[1] = sp->objPose[i][1];
      p[2] = sp->objPose[i][2];
    }
  }
  sync();
  // ---- lights (lane 0; positions of the positional lights are kept for the kilobots)
  const LightConst* lc = a.lights + (size_t)scene * (a.L.numLights > 0 ? a.L.numLights : 1);
  if (lane == 0) {
    int off = 0;
    for (int pos = 0; pos < NL; ++pos) {
      int c = 0;
#pragma unroll
      for (int q = 0; q < KB_MAX_LIGHTS; ++q)
        if (q == pos) c = order[q];
      const int type = lc[pos].type;
      if (type == KB_LIGHT_LINEAR) {
        light[off] = sp->lightInit[c][0];
        off += 1;
        continue;
      }
      double px, py;
      if (sp->lightMode[c] == 1) {
        double u0, u1;
        g.uniform2(KS_LIGHT, 4u * (uint32_t)pos, &u0, &u1);
        px = u0 * sp->sizeX + lox;
        py = u1 * sp->sizeY + loy;
      } else if (sp->lightMode[c] == 2 && M > 0) {
        double u0, u1;
        g.uniform2(KS_LIGHT, 4u * (uint32_t)pos + 1u, &u0, &u1);
        int which = (int)(u0 * (double)M);
        which = which >= M ? M - 1 : which;
        const double radius = 1.2 * sp->objExtent[which] / 2;
        const double angle = u1 * 2 * pi - pi;
        px = pose[3 * which + 0] + cos(angle) * radius;
        py = pose[3 * which + 1] + sin(angle) * radius;
      } else {
        px = sp->lightInit[c][0];
        py = sp->lightInit[c][1];
      }
      light[off] = px;
      light[off + 1] = py;
      if (type == KB_LIGHT_MOMENTUM) {
        double u0, u1;
        g.uniform2(KS_LIGHT, 4u * (uint32_t)pos + 2u, &u0, &u1);
        const double angle = u0 * 2 * pi - pi;
        light[off + 2] = sin(angle) * .01;
        light[off + 3] = cos(angle) * .01;
        off += 4;
      } else {
        off += 2;
      }
    }
  }
  sync();
  // ---- kilobots
  int npos = 0, posOff[KB_MAX_LIGHTS];
  {
    int off = 0;
    for (int pos = 0; pos < NL; ++pos) {
      const int type = lc[pos].type;
      if (type != KB_LIGHT_LINEAR) {
#pragma unroll
        for (int q = 0; q < KB_MAX_LIGHTS; ++q)
          if (q == npos) posOff[q] = off;
        ++npos;
      }
      off += type == KB_LIGHT_MOMENTUM ? 4 : (type == KB_LIGHT_LINEAR ? 1 : 2);
    }
  }
  int meanMode = sp->meanMode;
  if (meanMode == 1 && npos == 0) meanMode = 2;
  double rmx = 0.0, rmy = 0.0;
  if (meanMode == 2) {
    double u0, u1;
    g.uniform2(KS_SWARM, 0u, &u0, &u1);
    rmx = (u0 * sp->sizeX + lox) * 0.9;
    rmy = (u1 * sp->sizeY + loy) * 0.9;
  }
  for (int k = lane; k < N; k += nlanes) {
    double mx, my;
    if (meanMode == 1) {
      int pick = 0;
      if (npos > 1) {
        double u0, u1;
        g.uniform2(KS_SWARM, 1u + (uint32_t)k, &u0, &u1);
        pick = (int)(u0 * (double)npos);
        pick = pick >= npos ? npos - 1 : pick;
      }
      int o = 0;
#pragma unroll
      for (int q = 0; q < KB_MAX_LIGHTS; ++q)
        if (q == pick) o = posOff[q];
      mx = light[o];
      my = light[o + 1];
    } else if (meanMode == 2) {
      mx = rmx;
      my = rmy;
    } else {
      mx = sp->mean[0];
      my = sp->mean[1];
    }
    double z0, z1;
    g.normal2(KS_KILOBOT_POS, (uint32_t)k, &z0, &z1);
    double x = z0 * sp->std + mx, y = z1 * sp->std + my;
    x = fmax(x, lox + 0.02);
    y = fmax(y, loy + 0.02);
    x = fmin(x, -lox - 0.02);
    y = fmin(y, -loy - 0.02);
    double* p = pose + 3 * (Mmax + k);
    p[0] = x;
    p[1] = y;
    p[2] = 0.0;
  }
  sync();
  return scene;
}

}  // namespace kb
