// kb_b200.cu -- C-ABI (include/kb_b200.h) + kernels of the B200-native batched Kilobots step.
//
// Host side: turns the scene description into the device template (hull / normals / centroid /
// mass data exactly as Box2D 2.3.x derives them at fixture creation -- b2PolygonShape::Set,
// ComputeMass, b2Body::ResetMassData; reached from gym_kilobots/lib/body.py:136-142,187-192,
// 245-251), sizes the per-env state image, and launches one lane group per environment.
// There is no CPU fallback: without an sm_100 device kb_create fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "kb_step_kernel.cuh"
#include "kb_swarm.cuh"
#include "kb_render.cuh"
#include "kb_local.cuh"
#include "kb_jit.h"

namespace kb {

// ----------------------------------------------------------------------------------- kernels
// the generic step kernel: offsets, counts and constants come from the Layout in the kernel parameters
template <int LPE>
__global__ void __launch_bounds__(KB_STEP_BOUNDS(LPE)) kb_step_kernel(const __grid_constant__ KernelArgs a) {
  stepKernelBody<LPE>(a, a.L);
}

template <int LPE>
__global__ void __launch_bounds__(KB_BLOCK_OF(LPE)) kb_reset_kernel(const __grid_constant__ KernelArgs a) {
  constexpr int EPB = KB_BLOCK_OF(LPE) / LPE;
  const int slot = threadIdx.x / LPE;
  const int env = blockIdx.x * EPB + slot;
  const int envIn = min(env, a.numEnvs - 1);
  if (a.mask && !a.mask[envIn]) return;
  const Layout& L = a.L;
  Sim<LPE, false> s(a.L);
  s.g.init();
  s.bind(slot);
  s.blob = a.blobs + (size_t)env * L.blobWords;
  int scene = a.envScene ? a.envScene[envIn] : 0;
  if (a.sampler && env < a.numEnvs) {
    // a fresh scene for this env, drawn here: counter-based, keyed by (seed, global env id, episode)
    const uint32_t ep = a.episode[env];
    scene = sampleScene(a, env, scene, ep, s.g.lane, LPE, [&]() { s.g.sync(); });
    if (s.g.lane == 0) {
      a.episode[env] = ep + 1u;
      if (a.envSceneW) a.envSceneW[env] = scene;
    }
  }
  s.px = a.proxies + (size_t)scene * L.Pp;
  s.bc = a.bodies + (size_t)scene * L.Bp;
  s.lights = a.lights + (size_t)scene * (a.L.numLights > 0 ? a.L.numLights : 1);
  s.S = L.B;
  const int lane = s.g.lane;
  for (int i = lane; i < L.stateWords; i += LPE) s.word(i) = 0u;
  for (int i = lane; i < 2 * KB_NUM_COUNTERS; i += LPE) reinterpret_cast<uint32_t*>(s.blob)[L.oCnt + i] = 0u;
  s.g.sync();
  if (lane == 0) {
    s.hdr(H_NC) = 0u;
    s.hdr(H_STATUS) = 0u;
    s.hdr(H_SCENE) = (uint32_t)scene;
  }
  resetEnvLayer(s, a, env, envIn, lane, LPE);
  // bodies: b2World::CreateBody + CreateFixture (lib/body.py:32-38); an absent body (a padded index the scene does not
  // populate) in the canonical state whatever the pose input holds: zero pose and velocity, asleep, identity transform
  for (int b = lane; b < L.B; b += LPE) {
    if (__ldg(&s.bc[b].kind) == KB_BODY_ABSENT) {
      s.pos4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      s.vel4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      s.xf4(b) = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
      continue;
    }
    const double* p = a.pose + ((size_t)envIn * L.B + b) * 3;
    const float x = (float)(25.0 * p[0]);
    const float y = (float)(25.0 * p[1]);
    const float ang = (float)p[2];
    Xf xf;
    xf.p = mk(x, y);
    xf.q = rot_set(ang);
    const V2 lc = mk(__ldg(&s.bc[b].lcx), __ldg(&s.bc[b].lcy));
    const V2 c = xmul(xf, lc);
    s.pos4(b) = make_float4(c.x, c.y, ang, 0.0f);
    s.vel4(b) = make_float4(0.0f, 0.0f, 0.0f, u2f(BF_AWAKE));
    s.xf4(b) = make_float4(x, y, xf.q.s, xf.q.c);
  }
  s.g.sync();
  s.initScratch();
  // proxies: b2Fixture::CreateProxies -> fat AABB = aabb +- aabbExtension, buffered as moved
  uint32_t mlo = 0u, mhi = 0u;
  const int P = __ldg(&a.scenes[scene].numProxies);
  for (int p = lane; p < L.P; p += LPE) {
    if (p >= P) {
      s.fat4(p) = make_float4(3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f);  // unused slot: never overlaps
      continue;
    }
    const int b = __ldg(&s.px[p].body);
    V2 lo, hi;
    s.shapeAABB(p, s.bodyXf(b), &lo, &hi);
    s.fat4(p) = make_float4(lo.x - KB_AABB_EXTENSION, lo.y - KB_AABB_EXTENSION, hi.x + KB_AABB_EXTENSION,
                            hi.y + KB_AABB_EXTENSION);
    if (p < 32) mlo |= 1u << p; else mhi |= 1u << (p - 32);
  }
  mlo = s.g.red_or(mlo);
  mhi = s.g.red_or(mhi);
  if (lane == 0) {
    s.hdr(H_MOVED) = mlo;
    s.hdr(H_MOVED + 1) = mhi;
  }
  s.g.sync();
  s.findNewContacts();  // b2World::Step: m_flags & e_newFixture -> FindNewContacts
  s.worldStep();        // kilobots_env.py:157 "step to resolve"
  if (lane == 0 && a.status && env < a.numEnvs) a.status[env] = (int32_t)s.hdr(H_STATUS);
  s.storeState();
}

// Body.set_pose (lib/body.py:67-69) -> b2Body::SetTransform
template <int LPE>
__global__ void __launch_bounds__(KB_BLOCK_OF(LPE)) kb_setpose_kernel(const __grid_constant__ KernelArgs a) {
  constexpr int EPB = KB_BLOCK_OF(LPE) / LPE;
  const int slot = threadIdx.x / LPE;
  const int env = blockIdx.x * EPB + slot;
  const int envIn = min(env, a.numEnvs - 1);
  const Layout& L = a.L;
  Sim<LPE, false> s(a.L);
  s.g.init();
  s.bind(slot);
  s.blob = a.blobs + (size_t)env * L.blobWords;
  const int scene = a.envScene ? (int)reinterpret_cast<const uint32_t*>(s.blob)[L.oHdr + H_SCENE] : 0;
  s.px = a.proxies + (size_t)scene * L.Pp;
  s.bc = a.bodies + (size_t)scene * L.Bp;
  s.lights = a.lights + (size_t)scene * (a.L.numLights > 0 ? a.L.numLights : 1);
  s.S = L.B;
  s.loadState();
  s.initScratch();
  for (int b = s.g.lane; b <= L.B; b += LPE) s.isl(b) = -1;
  s.g.sync();
  for (int b = s.g.lane; b < L.B; b += LPE) {
    if (a.mask && !a.mask[(size_t)envIn * L.B + b]) continue;   // Body.set_pose touches this one body only
    if (s.bkind(b) == KB_BODY_ABSENT) continue;
    const double* p = a.pose + ((size_t)envIn * L.B + b) * 3;
    const float x = (float)(p[0] * 25.0);
    const float y = (float)(p[1] * 25.0);
    const float ang = (float)p[2];
    Xf xf;
    xf.q = rot_set(ang);
    xf.p = mk(x, y);
    const float4 k = s.bc4(b);
    const V2 c = xmul(xf, mk(k.z, k.w));
    float4 pos = s.pos4(b);
    pos.x = c.x; pos.y = c.y; pos.z = ang;
    s.pos4(b) = pos;
    s.xf4(b) = make_float4(x, y, xf.q.s, xf.q.c);
    s.sweep4(b) = make_float4(c.x, c.y, ang, 0.0f);
    s.oldq(b) = make_float2(xf.q.s, xf.q.c);
    s.isl(b) = 0;
  }
  s.g.sync();
  // SetTransform: Synchronize(xf, xf) with zero displacement.  xf1 == xf2 requires xf1.p == xf.p, which
  // synchronizeFixtures rebuilds as c0 - q*lc; SetTransform passes m_xf for both, so use toiMode=false
  // with the saved rotation and accept p = c - q*lc (identical for every body whose xf was synchronised).
  s.synchronizeFixtures(false);
  s.storeState();
}

// kb_current_scenes: the header word H_SCENE of every env's blob (the scene it was last reset with)
__global__ void kb_current_scenes_kernel(const float* __restrict__ blobs, int blobWords, int word, int numEnvs,
                                         int32_t* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < numEnvs) out[e] = (int32_t)reinterpret_cast<const uint32_t*>(blobs)[(size_t)e * blobWords + word];
}

// Episode statistics of a rank, reduced on the device to KB_REDUCED_STATS doubles (the operand of the NCCL
// all-reduce in KilobotsVecEnv.all_reduce_episode_stats).  One block, fixed summation tree: the result depends
// on E only, never on scheduling.
__global__ void __launch_bounds__(1024) kb_reduce_stats_kernel(const double* task, const float* blobs, int blobWords,
                                                                int statusWord, int numEnvs, double* out) {
  __shared__ double sh[KB_REDUCED_STATS][32];
  double acc[KB_REDUCED_STATS];
  for (int k = 0; k < KB_REDUCED_STATS; ++k) acc[k] = 0.0;
  for (int e = threadIdx.x; e < numEnvs; e += blockDim.x) {
    const double* ts = task + (size_t)e * KB_TASK_WORDS + 3;
    acc[0] += 1.0;
    for (int k = 0; k < KB_EPISODE_STATS; ++k) acc[1 + k] += ts[k];
    acc[7] += reinterpret_cast<const uint32_t*>(blobs)[(size_t)e * blobWords + statusWord] != 0u ? 1.0 : 0.0;
  }
  for (int k = 0; k < KB_REDUCED_STATS; ++k) {
    double v = acc[k];
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, d);
    if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    for (int k = 0; k < KB_REDUCED_STATS; ++k) {
      double v = threadIdx.x < (blockDim.x >> 5) ? sh[k][threadIdx.x] : 0.0;
      for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, d);
      if (threadIdx.x == 0) out[k] = v;
    }
  }
}

// ------------------------------------------------------------------------------- host state
struct Handle {
  int device = 0;
  int numEnvs = 0, numScenes = 0;
  Layout L;
  std::vector<std::vector<BodyConst>> hostBodies;  // per scene
  std::vector<int> hostNumProxies;                  // per scene
  std::vector<int> hostNumObjects, hostNumKilobots; // per scene (L.M / L.N are the maxima over the scenes)
  float* dBlobs = nullptr;
  int32_t* dEnvScene = nullptr;
  ProxyConst* dProxies = nullptr;
  BodyConst* dBodies = nullptr;
  SceneConst* dScenes = nullptr;
  LightConst* dLights = nullptr;
  // staging for kb_step_host
  double* dAction = nullptr;
  // kb_step_host staging: ONE device allocation, sections at hostOff[] (see kb_get_host_layout)
  uint8_t* dOut = nullptr;
  int64_t hostOff[6] = {0, 0, 0, 0, 0, 0}, hostTotal = 0;
  float *dObsK = nullptr, *dObsO = nullptr, *dReward = nullptr;
  double* dObsL = nullptr;
  uint8_t* dDone = nullptr;
  int32_t* dStatus = nullptr;
  float wall[4] = {0.0f, 0.0f, 0.0f, 0.0f};   // table rectangle x0 y0 x1 y1, b2 units (render window)
  int32_t* dRenderIds = nullptr;
  int renderIdsCap = 0;
  // task layer (extension)
  TaskConst task = {};
  double* dTask = nullptr;   // [E][KB_TASK_WORDS]
  float* obsFlat = nullptr;  // caller-owned device buffer bound by kb_bind_flat_observation
  int envsPerBlock = 4;
  size_t smemBytes = 0;
  SwarmLayout W = {};          // W.enabled: the large-swarm tier (kb_swarm.cuh) runs this batch
  // kb_step_host pipeline: chunks of the batch alternate between two side streams, so that the device->host copy of
  // one chunk overlaps the kernel of the next
  // on-device scene sampling at reset (kb_sample.cuh)
  SamplerConst* dSampler = nullptr;             // [KB_SAMPLE_MAX_CONFIGS], numConfigs of them set
  double *dSamplePose = nullptr, *dSampleLight = nullptr;
  uint32_t* dEpisode = nullptr;
  int numConfigs = 0;
  std::vector<int> hostSceneConfig;              // configuration of each scene (-1 = none)
  int32_t* dSceneConfig = nullptr;               // [numScenes]
  double* dConfigCdf = nullptr;                  // [KB_SAMPLE_MAX_CONFIGS]
  bool weighted = false;
  cudaStream_t pipe[2] = {nullptr, nullptr};
  cudaEvent_t evFork = nullptr, evJoin[2] = {nullptr, nullptr};
  int hostChunks = 1;
  // the step kernel compiled for this batch's layout (kb_jit.h); null: the generic kb_step_kernel<LPE> runs
  cudaKernel_t stepJit = nullptr;
  float jitMs = 0.0f;          // its compile time in kb_create (0: from a cache)
  std::string jitReason;       // why the generic kernel runs instead
#ifdef KB_PROFILE
  unsigned long long* dProf = nullptr;
#endif
};

static int launchGrid(const Handle* h) { return (h->numEnvs + h->envsPerBlock - 1) / h->envsPerBlock; }

// The dynamic shared-memory limit is an attribute of the kernel, shared by every handle of the process: only ever raise
// it, so that a batch created later with a smaller image (same kernel, fewer bodies) does not break an earlier one.
template <class K>
static cudaError_t raiseSmemLimit(K* kernel, size_t bytes) {
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
  if (e != cudaSuccess || (size_t)fa.maxDynamicSharedSizeBytes >= bytes) return e;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                             \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) return fail(KB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// --- Box2D fixture preprocessing (float32, same operation order as Box2D) ---------------------
struct HV2 {
  float x, y;
};
static inline HV2 hv(float x, float y) { return HV2{x, y}; }
static inline HV2 operator+(HV2 a, HV2 b) { return hv(a.x + b.x, a.y + b.y); }
static inline HV2 operator-(HV2 a, HV2 b) { return hv(a.x - b.x, a.y - b.y); }
static inline HV2 operator*(float s, HV2 a) { return hv(s * a.x, s * a.y); }
static inline float hdot(HV2 a, HV2 b) { return a.x * b.x + a.y * b.y; }
static inline float hcross(HV2 a, HV2 b) { return a.x * b.y - a.y * b.x; }

// b2PolygonShape::Set: weld, gift-wrap from the right-most vertex, normals, centroid
static bool buildPolygon(const KbFixtureDef& fd, ProxyConst* pc) {
  const float linearSlop = 0.005f;
  int n = std::min(fd.vertex_count, (int)KB_MAX_POLY_VERTS);
  HV2 ps[KB_MAX_POLY_VERTS];
  int tempCount = 0;
  for (int i = 0; i < n; ++i) {
    HV2 v = hv(fd.vx[i], fd.vy[i]);
    bool unique = true;
    for (int j = 0; j < tempCount; ++j) {
      HV2 d = v - ps[j];
      if (hdot(d, d) < 0.5f * linearSlop) {
        unique = false;
        break;
      }
    }
    if (unique) ps[tempCount++] = v;
  }
  n = tempCount;
  if (n < 3) return false;
  int i0 = 0;
  float x0 = ps[0].x;
  for (int i = 1; i < n; ++i) {
    float x = ps[i].x;
    if (x > x0 || (x == x0 && ps[i].y < ps[i0].y)) {
      i0 = i;
      x0 = x;
    }
  }
  int hull[KB_MAX_POLY_VERTS];
  int m = 0;
  int ih = i0;
  for (;;) {
    hull[m] = ih;
    int ie = 0;
    for (int j = 1; j < n; ++j) {
      if (ie == ih) {
        ie = j;
        continue;
      }
      HV2 r = ps[ie] - ps[hull[m]];
      HV2 v = ps[j] - ps[hull[m]];
      float c = hcross(r, v);
      if (c < 0.0f) ie = j;
      if (c == 0.0f && hdot(v, v) > hdot(r, r)) ie = j;
    }
    ++m;
    ih = ie;
    if (ie == i0) break;
  }
  pc->count = m;
  for (int i = 0; i < m; ++i) {
    pc->vx[i] = ps[hull[i]].x;
    pc->vy[i] = ps[hull[i]].y;
  }
  for (int i = 0; i < m; ++i) {
    int i2 = i + 1 < m ? i + 1 : 0;
    HV2 edge = hv(pc->vx[i2], pc->vy[i2]) - hv(pc->vx[i], pc->vy[i]);
    // b2Cross(edge, 1) then Normalize
    HV2 nrm = hv(1.0f * edge.y, -1.0f * edge.x);
    float len = sqrtf(nrm.x * nrm.x + nrm.y * nrm.y);
    if (!(len < FLT_EPSILON)) {
      float inv = 1.0f / len;
      nrm.x *= inv;
      nrm.y *= inv;
    }
    pc->nx[i] = nrm.x;
    pc->ny[i] = nrm.y;
  }
  // ComputeCentroid (reference point at the origin)
  HV2 c = hv(0.0f, 0.0f);
  float area = 0.0f;
  const float inv3 = 1.0f / 3.0f;
  for (int i = 0; i < m; ++i) {
    HV2 p1 = hv(0.0f, 0.0f);
    HV2 p2 = hv(pc->vx[i], pc->vy[i]);
    HV2 p3 = i + 1 < m ? hv(pc->vx[i + 1], pc->vy[i + 1]) : hv(pc->vx[0], pc->vy[0]);
    HV2 e1 = p2 - p1;
    HV2 e2 = p3 - p1;
    float D = hcross(e1, e2);
    float triangleArea = 0.5f * D;
    area += triangleArea;
    c = c + (triangleArea * inv3) * ((p1 + p2) + p3);
  }
  c = (1.0f / area) * c;
  pc->cx = c.x;
  pc->cy = c.y;
  return true;
}

static void buildBox(float hx, float hy, ProxyConst* pc) {
  pc->count = 4;
  const float vx[4] = {-hx, hx, hx, -hx}, vy[4] = {-hy, -hy, hy, hy};
  const float nx[4] = {0.0f, 1.0f, 0.0f, -1.0f}, ny[4] = {-1.0f, 0.0f, 1.0f, 0.0f};
  for (int i = 0; i < 4; ++i) {
    pc->vx[i] = vx[i];
    pc->vy[i] = vy[i];
    pc->nx[i] = nx[i];
    pc->ny[i] = ny[i];
  }
  pc->cx = 0.0f;
  pc->cy = 0.0f;
}

// b2Shape::ComputeMass
static void fixtureMass(const ProxyConst& pc, float density, float* mass, HV2* center, float* I) {
  const float b2pi = 3.14159265359f;
  if (pc.type == SHAPE_CIRCLE) {
    *mass = density * b2pi * pc.radius * pc.radius;
    *center = hv(0.0f, 0.0f);
    *I = *mass * (0.5f * pc.radius * pc.radius + hdot(*center, *center));
    return;
  }
  HV2 ctr = hv(0.0f, 0.0f);
  float area = 0.0f, inertia = 0.0f;
  HV2 s = hv(0.0f, 0.0f);
  for (int i = 0; i < pc.count; ++i) s = s + hv(pc.vx[i], pc.vy[i]);
  s = (1.0f / pc.count) * s;
  const float k_inv3 = 1.0f / 3.0f;
  for (int i = 0; i < pc.count; ++i) {
    HV2 e1 = hv(pc.vx[i], pc.vy[i]) - s;
    HV2 e2 = i + 1 < pc.count ? hv(pc.vx[i + 1], pc.vy[i + 1]) - s : hv(pc.vx[0], pc.vy[0]) - s;
    float D = hcross(e1, e2);
    float triangleArea = 0.5f * D;
    area += triangleArea;
    ctr = ctr + (triangleArea * k_inv3) * (e1 + e2);
    float ex1 = e1.x, ey1 = e1.y, ex2 = e2.x, ey2 = e2.y;
    float intx2 = ex1 * ex1 + ex2 * ex1 + ex2 * ex2;
    float inty2 = ey1 * ey1 + ey2 * ey1 + ey2 * ey2;
    inertia += (0.25f * k_inv3 * D) * (intx2 + inty2);
  }
  *mass = density * area;
  ctr = (1.0f / area) * ctr;
  *center = ctr + s;
  *I = density * inertia;
  *I += *mass * (hdot(*center, *center) - hdot(ctr, ctr));
}

static int lightStateDim(int type) { return type == KB_LIGHT_MOMENTUM ? 4 : (type == KB_LIGHT_LINEAR ? 1 : 2); }
static int lightActionDim(int type) { return type == KB_LIGHT_LINEAR ? 1 : 2; }
static int round4(int x) { return (x + 3) & ~3; }

// type, radius and geometry of a fixture's proxy
static int buildFixtureShape(const KbFixtureDef& fd, ProxyConst* out) {
  ProxyConst& pc = *out;
  if (fd.shape == KB_SHAPE_CIRCLE) {
    pc.type = SHAPE_CIRCLE;
    pc.radius = fd.radius;
  } else if (fd.shape == KB_SHAPE_BOX) {
    pc.type = SHAPE_POLYGON;
    pc.radius = 2.0f * 0.005f;
    buildBox(fd.hx, fd.hy, &pc);
  } else if (fd.shape == KB_SHAPE_POLYGON) {
    pc.type = SHAPE_POLYGON;
    pc.radius = 2.0f * 0.005f;
    if (!buildPolygon(fd, &pc)) return fail(KB_ERR_INVALID, "degenerate polygon fixture");
  } else {
    return fail(KB_ERR_INVALID, "unknown fixture shape");
  }
  return KB_OK;
}

// child i of the table chain, kilobots_env.py:46-51: (x0,y1) -> (x0,y0) -> (x1,y0) -> (x1,y1) [-> (x0,y1)], with the ghost
// vertices of b2ChainShape::GetChildEdge.  pc is zeroed; body and friction are the caller's.
static void buildChainEdge(const KbSceneDesc& sd, int i, ProxyConst* out) {
  const float vx[5] = {sd.wall_x0, sd.wall_x0, sd.wall_x1, sd.wall_x1, sd.wall_x0};
  const float vy[5] = {sd.wall_y1, sd.wall_y0, sd.wall_y0, sd.wall_y1, sd.wall_y1};
  const bool loop = sd.wall_edges == 4;
  const int count = loop ? 5 : 4;
  ProxyConst& pc = *out;
  pc.type = SHAPE_EDGE;
  pc.radius = 2.0f * 0.005f;
  pc.restitution = 0.0f;
  pc.vx[1] = vx[i]; pc.vy[1] = vy[i];
  pc.vx[2] = vx[i + 1]; pc.vy[2] = vy[i + 1];
  if (i > 0) { pc.vx[0] = vx[i - 1]; pc.vy[0] = vy[i - 1]; pc.has0 = 1; }
  else if (loop) { pc.vx[0] = vx[count - 2]; pc.vy[0] = vy[count - 2]; pc.has0 = 1; }
  if (i < count - 2) { pc.vx[3] = vx[i + 2]; pc.vy[3] = vy[i + 2]; pc.has3 = 1; }
  else if (loop) { pc.vx[3] = vx[1]; pc.vy[3] = vy[1]; pc.has3 = 1; }
}

// The scene's bodies in the batch's padded layout: object j at body index j, kilobot k at Mmax + k; the other indices
// up to B = Bp - 1 are absent bodies (kind KB_BODY_ABSENT, no proxy, zero mass data).  Proxies are numbered as in a
// compact world of the scene's own bodies: the table edges, then the fixtures of the present bodies in body order.
static int buildScene(const KbSceneDesc& sd, int Mmax, int Bp, int Pp, std::vector<ProxyConst>* proxies,
                      std::vector<BodyConst>* bodies, SceneConst* sc) {
  const int B = Bp - 1;   // the static table's slot
  proxies->assign(Pp, ProxyConst());
  bodies->assign(Bp, BodyConst());
  std::memset(proxies->data(), 0, sizeof(ProxyConst) * Pp);
  std::memset(bodies->data(), 0, sizeof(BodyConst) * Bp);
  int p = 0;
  if (sd.wall_edges != 0 && sd.wall_edges != 3 && sd.wall_edges != 4) return fail(KB_ERR_INVALID, "wall_edges must be 0, 3 or 4");
  for (int i = 0; i < sd.wall_edges; ++i) {
    ProxyConst& pc = (*proxies)[p++];
    pc.body = B;  // static slot
    pc.friction = sd.wall_friction;
    buildChainEdge(sd, i, &pc);
  }
  for (int b = 0; b < B; ++b) (*bodies)[b].kind = KB_BODY_ABSENT;
  for (int be = 0; be < sd.num_bodies; ++be) {
    const KbBodyDef& bd = sd.bodies[be];
    const int b = be < sd.num_objects ? be : Mmax + (be - sd.num_objects);
    BodyConst& bcst = (*bodies)[b];
    if (bd.num_fixtures < 1 || bd.num_fixtures > KB_MAX_FIXTURES) return fail(KB_ERR_INVALID, "body needs 1..3 fixtures");
    bcst.kind = bd.kind;
    bcst.firstProxy = p;
    bcst.numProxies = bd.num_fixtures;
    bcst.linearDamping = bd.linear_damping;
    bcst.angularDamping = bd.angular_damping;
    // SimplePhototaxisKilobot.step sets linearDamping = 0 on every call (lib/kilobot.py:203); the only
    // step that runs before the first call is reset's settle step, where the velocity is zero.
    if (bd.kind == KB_KILOBOT_SIMPLE_PHOTOTAXIS) bcst.linearDamping = 0.0f;
    for (int f = 0; f < bd.num_fixtures; ++f) {
      const KbFixtureDef& fd = bd.fixtures[f];
      ProxyConst& pc = (*proxies)[p++];
      pc.body = b;
      pc.friction = fd.friction;
      pc.restitution = fd.restitution;
      const int rc = buildFixtureShape(fd, &pc);
      if (rc != KB_OK) return rc;
    }
    // b2Body::ResetMassData: fixtures are visited newest first (m_fixtureList is LIFO)
    float mass = 0.0f, I = 0.0f;
    HV2 lc = hv(0.0f, 0.0f);
    for (int f = bd.num_fixtures - 1; f >= 0; --f) {
      const float density = bd.fixtures[f].density;
      if (density == 0.0f) continue;
      float m, i;
      HV2 c;
      fixtureMass((*proxies)[bcst.firstProxy + f], density, &m, &c, &i);
      mass += m;
      lc = lc + m * c;
      I += i;
    }
    float invMass, invI;
    if (mass > 0.0f) {
      invMass = 1.0f / mass;
      lc = invMass * lc;
    } else {
      mass = 1.0f;
      invMass = 1.0f;
    }
    if (I > 0.0f) {
      I -= mass * hdot(lc, lc);
      invI = 1.0f / I;
    } else {
      invI = 0.0f;
    }
    bcst.invMass = invMass;
    bcst.invI = invI;
    bcst.lcx = lc.x;
    bcst.lcy = lc.y;
  }
  sc->numProxies = p;
  for (int q = p; q < Pp; ++q) {  // unused slots (scenes with fewer fixtures): inert table proxies that never overlap
    (*proxies)[q].body = B;
    (*proxies)[q].type = SHAPE_EDGE;
  }
  sc->wallEdges = sd.wall_edges;
  sc->rewardConst = sd.reward_const;
  sc->numObjects = (int16_t)sd.num_objects;
  sc->numKilobots = (int16_t)(sd.num_bodies - sd.num_objects);
  return KB_OK;
}

static void fillArgs(const Handle* h, KernelArgs* a) {
  std::memset(a, 0, sizeof(*a));
  a->L = h->L;
  a->W = h->W;
  a->blobs = h->dBlobs;
  a->envScene = h->dEnvScene;
  a->proxies = h->dProxies;
  a->bodies = h->dBodies;
  a->scenes = h->dScenes;
  a->lights = h->dLights;
  a->numEnvs = h->numEnvs;
  a->task = h->task;
  a->taskState = h->dTask;
#ifdef KB_PROFILE
  a->prof = h->dProf;
#endif
}

// The batch's layout (h->L, h->W), tier, lane width and shared-memory size from its scenes.  Needs no device: `prop`
// only sizes the large-swarm tier's image.
static int planBatch(const KbSceneDesc* scenes, int32_t num_scenes, int32_t max_contacts, const cudaDeviceProp& prop,
                     Handle* h) {
  const KbSceneDesc& s0 = scenes[0];
  // padded body layout: M / N are the largest object / kilobot counts over the scenes, objects at 0..M-1, kilobots at
  // M..M+N-1; a scene with fewer leaves absent bodies at the indices it does not populate
  int M = 0, N = 0;
  for (int s = 0; s < num_scenes; ++s) {
    const KbSceneDesc& sd = scenes[s];
    if (sd.num_bodies < 1 || sd.num_objects < 0 || sd.num_objects > sd.num_bodies || sd.num_bodies > 0xFFFF || !sd.bodies)
      return fail(KB_ERR_INVALID, "kb_create: bad body counts");
    M = std::max(M, (int)sd.num_objects);
    N = std::max(N, (int)(sd.num_bodies - sd.num_objects));
  }
  const int B = M + N;
  // tier: the lane-group kernels (kb_step.cuh) hold up to 62 bodies; above that -- or on request (KB_FORCE_SWARM=1, used
  // by the tests to cross-check the two tiers on the same scenes) -- the CTA-per-env swarm tier (kb_swarm.cuh)
  bool swarm = B > KB_MAX_BODIES;
  if (const char* ev = getenv("KB_FORCE_SWARM")) swarm = swarm || atoi(ev) != 0;
  if (swarm) {
    if (B > KB_SWARM_MAX_BODIES) return fail(KB_ERR_CAPACITY, "kb_create: more than 2040 bodies per env is not supported");
    if (M != 0) return fail(KB_ERR_CAPACITY, "kb_create: the large-swarm tier (> 62 bodies per env) supports kilobots only (no pushable objects)");
    for (int s = 0; s < num_scenes; ++s)
      for (int b = 0; b < scenes[s].num_bodies; ++b) {
        const KbBodyDef& bd = scenes[s].bodies[b];
        if (bd.kind == KB_BODY_OBJECT || bd.num_fixtures != 1 || bd.fixtures[0].shape != KB_SHAPE_CIRCLE ||
            bd.fixtures[0].friction != 0.0f || bd.fixtures[0].restitution != 0.0f || !(bd.fixtures[0].density > 0.0f))
          return fail(KB_ERR_CAPACITY, "kb_create: the large-swarm tier needs every body to be a kilobot (one frictionless circle fixture)");
      }
  }
  if (s0.num_lights > KB_MAX_LIGHTS) return fail(KB_ERR_INVALID, "kb_create: too many lights");
  int P = 0;
  for (int s = 0; s < num_scenes; ++s) {
    const KbSceneDesc& sd = scenes[s];
    if (sd.num_lights != s0.num_lights ||
        sd.steps_per_action != s0.steps_per_action || sd.velocity_iterations != s0.velocity_iterations ||
        sd.position_iterations != s0.position_iterations || sd.dt != s0.dt || sd.damping_mode != s0.damping_mode ||
        sd.enable_toi != s0.enable_toi || sd.enable_sleep != s0.enable_sleep)
      return fail(KB_ERR_INVALID, "kb_create: scenes must agree in light counts and simulation constants");
    {
      // light components may differ between scenes (a shuffled CompositeLight, different radii): the constants are
      // held per scene; the state / action vectors must have the same total length
      int sl = 0, al = 0, sl0 = 0, al0 = 0;
      for (int l = 0; l < sd.num_lights; ++l) {
        sl += lightStateDim(sd.lights[l].type); al += lightActionDim(sd.lights[l].type);
        sl0 += lightStateDim(s0.lights[l].type); al0 += lightActionDim(s0.lights[l].type);
      }
      if (sl != sl0 || al != al0) return fail(KB_ERR_INVALID, "kb_create: scenes must agree in light state / action dimensions");
    }
    int p = sd.wall_edges;
    for (int b = 0; b < sd.num_bodies; ++b) p += sd.bodies[b].num_fixtures;
    P = std::max(P, p);
    // body kinds agree at every padded index that two scenes both populate
    for (int t = 0; t < s; ++t) {
      const KbSceneDesc& st = scenes[t];
      const int mo = std::min(sd.num_objects, st.num_objects);
      const int nk = std::min(sd.num_bodies - sd.num_objects, st.num_bodies - st.num_objects);
      bool same = true;
      for (int b = 0; b < mo; ++b) same = same && sd.bodies[b].kind == st.bodies[b].kind;
      for (int k = 0; k < nk; ++k) same = same && sd.bodies[sd.num_objects + k].kind == st.bodies[st.num_objects + k].kind;
      if (!same) return fail(KB_ERR_INVALID, "kb_create: scenes must agree in body kinds");
    }
  }
  if (!swarm && P > KB_MAX_PROXIES) return fail(KB_ERR_CAPACITY, "kb_create: more than 64 proxies per env is not supported");

  Layout& L = h->L;
  std::memset(&L, 0, sizeof(L));
  L.B = B; L.M = M; L.N = N; L.P = P;
  L.Bp = B + 1;
  L.Pp = P;
  L.numLights = s0.num_lights;
  for (int l = 0; l < s0.num_lights; ++l) {
    L.L += lightStateDim(s0.lights[l].type);
    L.A += lightActionDim(s0.lights[l].type);
  }
  if (swarm) {
    SwarmLayout& W = h->W;
    W.enabled = 1;
    // capacities: the caller's, else 8B + 32 persistent pairs and 3B + 32 touching contacts (hexagonal packing) --
    // shrunk step by step (never below 5B + 32 / 2B + 32) until the CTA's image fits the SM's shared memory
    int cmaxTry = round4(max_contacts > 0 ? max_contacts : std::min(P * (P - 1) / 2, 8 * B + 32));
    if (cmaxTry > 65532) cmaxTry = 65532;                       // 16-bit contact indices in the schedule
    // (an explicit max_contacts also sizes the solver: stacked spawns touch more than 3 neighbours per body)
    int kmaxTry = round4(std::min(cmaxTry, max_contacts > 0 ? max_contacts : 3 * B + 32));
    for (;;) {
    L.Cmax = cmaxTry;
    L.Kmax = kmaxTry;
    L.Gmax = 0;
    L.KW = 0;
    W.movedWords = round4((P + 31) / 32);
    int o = 0;
    L.oHdr = o; o += H_WORDS;
    L.oLight = o; o += round4(2 * std::max(L.L, 1));
    L.oPos = o; o += 4 * L.Bp;
    L.oVel = o; o += 4 * L.Bp;
    L.oXf = o; o += 4 * L.Bp;
    L.oFat = o; o += 4 * L.Pp;
    L.stateWords = round4(o);
    W.oMoved = o; o += W.movedWords;
    L.oCw = o; o += L.Cmax;
    W.oCpair = o; o += L.Cmax;
    L.oCnt = o; o += 2 * KB_NUM_COUNTERS;
    L.oCtrl = o; o += round4(8 * std::max(N, 1));
    L.oMan = o; o += SR_WORDS * L.Cmax;
    W.oSweep = o; o += 4 * L.Bp;
    L.oToi = o; o += L.Cmax;
    L.oGen = o;
    const int K = L.Kmax;
    W.oEnt0 = o; o += K;
    W.oEntC = o; o += round4((K + 1) / 2);
    W.oEntI = o; o += round4((K + 1) / 2);
    W.oRow = o; o += round4((K + 4 + 1) / 2);
    W.oRec = round4(o); o = W.oRec + 12 * K;
    W.oTlC = o; o += round4((K + 1) / 2);
    W.hashSize = 64;
    W.hashShift = 26;
    while (W.hashSize < L.Cmax + L.Cmax / 2) { W.hashSize *= 2; W.hashShift -= 1; }   // load factor <= 2/3 at capacity
    W.oHash = o; o += W.hashSize;
    L.blobWords = round4(o);
    auto al = [](int x, int a) { return (x + a - 1) / a * a; };
    int z = 0;
    W.zPos = z; z += 16 * L.Bp;
    W.zVel = z; z += 16 * L.Bp;
    W.zHdr = z; z += 4 * H_WORDS;
    W.zMoved = z; z += 4 * W.movedWords;
    z = al(z, 8);
    W.zLight = z; z += 8 * std::max(L.L, 1);
    W.zLc = z; z += 4 * LC_WORDS * std::max((int)s0.num_lights, 1);
    W.zMisc = z; z += 4 * 64;
    W.zIsl = z; z += al(2 * L.Bp, 4);
    W.zIslState = z; z += al(L.Bp, 4);
    z = al(z, 16);
    W.zDummy = z; z += 16 * 32;      // one row per lane: what the idle lanes of the solver relay load from and store to
    W.zScr = z;
    int q = 0;
    W.sTlB = q; q += 4 * K;
    W.sAdj = q; q += 8 * K;          // two packed entries (list index | other body << 16) per touching contact
    W.sBstart = q; q += al(2 * (L.Bp + 2), 4);
    W.sBcur = q; q += al(2 * (L.Bp + 2), 4);
    W.sOrd = q; q += al(2 * K, 4);
    W.sOlvl = q; q += al(2 * K, 4);
    W.sOisl = q; q += al(2 * K, 4);
    W.sStack = q; q += al(2 * L.Bp, 4);
    W.sBw = q; q += 4 * L.Bp;
    W.sLvlCnt = q; q += al(2 * (K + 4), 4);
    int scratch = q;
    W.cWakeAt = 0;
    scratch = std::max(scratch, 4 * L.Bp);
    // uniform grid over the table rectangle (+2 cells of margin), cell = 0.05 m (SURVEY 8d) = 1.25 b2 units
    const float cell = 1.25f;
    W.invCell = 1.0f / cell;
    W.gx0 = std::min(s0.wall_x0, s0.wall_x1) - 2.0f * cell;
    W.gy0 = std::min(s0.wall_y0, s0.wall_y1) - 2.0f * cell;
    W.gx = std::min(256, std::max(1, (int)std::ceil(std::fabs(s0.wall_x1 - s0.wall_x0) / cell) + 4));
    W.gy = std::min(256, std::max(1, (int)std::ceil(std::fabs(s0.wall_y1 - s0.wall_y0) / cell) + 4));
    q = 0;
    W.gCellStart = q; q += 4 * (W.gx * W.gy + 2);
    W.gCellCur = q;
    W.gSorted = q; q += al(2 * L.Pp, 4);
    W.gPcnt = q; q += 4 * L.Pp;
    q = al(q, 16);
    W.gFat = q; q += 16 * L.Pp;      // the fat AABBs, staged for the candidate tests (27 per proxy)
    W.gCand = q; q += 2 * 12 * std::min(512, al(L.Pp, 32));   // per live thread: the partners whose fat AABBs overlap (KB_SW_CAND u16 each)
    scratch = std::max(scratch, q);
    W.smemBytes = al(W.zScr + scratch, 16);
    if ((size_t)W.smemBytes <= (size_t)prop.sharedMemPerBlockOptin) break;
    const int kFloor = round4(2 * B + 32), cFloor = round4(5 * B + 32);   // (floors on the rounded values: the loop ends)
    if (kmaxTry > kFloor) kmaxTry = std::max(kFloor, round4(kmaxTry - B / 4 - 4));
    else if (max_contacts <= 0 && cmaxTry > cFloor) cmaxTry = std::max(cFloor, round4(cmaxTry - B / 2 - 4));
    else break;   // reported below: does not fit
    }
    {
      // threads per CTA: as many CTAs per SM as shared memory holds, each as wide as the register file then allows
      const int perSm = std::max(1, (int)((size_t)prop.sharedMemPerMultiprocessor / ((size_t)W.smemBytes + 1024)));
      L.lanesPerEnv = perSm >= 4 ? 128 : (perSm >= 2 ? 256 : 512);
      if (const char* ev = getenv("KB_SWARM_THREADS")) {
        const int v = atoi(ev);
        if (v == 128 || v == 256 || v == 512) L.lanesPerEnv = v;
      }
    }
    L.smemWords = W.smemBytes / 4;
  } else {
  // max_contacts > 0: the caller's capacity; 0: the throughput default (8B + 32 persistent pairs, 3B + 9 touching
  // contacts per solve: enough for separated swarms); < 0: every proxy pair, i.e. no pair can ever be dropped
  // (what the E = 1 drop-in facade asks for: the reference's clipped-Gaussian spawn may stack kilobots)
  const bool fullCapacity = max_contacts < 0;
  L.Cmax = round4(max_contacts > 0 ? max_contacts : (fullCapacity ? std::max(P * (P - 1) / 2, 4) : std::min(P * (P - 1) / 2, 8 * B + 32)));
  if (L.Cmax > 65535) L.Cmax = 65532;
  L.Kmax = round4(std::min(fullCapacity ? L.Cmax : std::min(L.Cmax, 3 * B + 9), (int)KB_MAX_SOLVER));
  L.KW = round4((L.Kmax + 31) / 32);  // words per body mask over the touching list, padded to whole 128-bit loads
  {
    // general constraints can only arise between proxies that are not frictionless circles-with-zero-restitution
    // partners; a safe bound is every pair of object proxies plus object proxies against the table edges.  The
    // TOI mini-island (one body against the table) uses the same records.
    int maxObjProxies = 0, maxWall = 0;
    for (int s = 0; s < num_scenes; ++s) {
      int op = 0;
      for (int b = 0; b < scenes[s].num_objects; ++b) op += scenes[s].bodies[b].num_fixtures;
      maxObjProxies = std::max(maxObjProxies, op);
      maxWall = std::max(maxWall, (int)scenes[s].wall_edges);
    }
    bool allKilobotsFrictionless = true;
    for (int s = 0; s < num_scenes; ++s)
      for (int b = scenes[s].num_objects; b < scenes[s].num_bodies; ++b)
        for (int f = 0; f < scenes[s].bodies[b].num_fixtures; ++f) {
          const KbFixtureDef& fd = scenes[s].bodies[b].fixtures[f];
          if (fd.friction != 0.0f || fd.restitution != 0.0f || fd.shape != KB_SHAPE_CIRCLE) allKilobotsFrictionless = false;
        }
    int gen = maxObjProxies * (maxObjProxies - 1) / 2 + maxObjProxies * maxWall;
    if (!allKilobotsFrictionless) gen = L.Kmax;
    L.Gmax = std::min(std::min(L.Kmax, 252), std::max(8, gen));   // general slots are 8-bit (sGs)
  }
  int o = 0;
  L.oHdr = o; o += H_WORDS;
  L.oLight = o; o += round4(2 * std::max(L.L, 1));
  L.oPos = o; o += 4 * L.Bp;
  L.oVel = o; o += 4 * L.Bp;
  L.oXf = o; o += 4 * L.Bp;
  L.oFat = o; o += 4 * L.Pp;
  L.oCw = o; o += L.Cmax;
  L.stateWords = round4(o);
  o = L.stateWords;
  L.oCnt = o; o += 2 * KB_NUM_COUNTERS;
  L.oCtrl = o; o += round4(8 * std::max(N, 1));
  L.oMan = o; o += MR_WORDS * L.Cmax;
  L.oGen = o; o += GR_WORDS * L.Gmax;
  L.oToi = o; o += L.Cmax;
  L.blobWords = round4(o);
  o = L.stateWords;
  L.sSweep = o; o += 4 * L.Bp;
  L.sOldQ = o; o += round4(2 * L.Bp);
  L.sBc = o; o += 4 * L.Bp;
  L.sIsl = o; o += round4(L.Bp);
  L.sIslFlag = o; o += round4(L.Bp);
  L.sStack = o; o += round4(L.Bp);
  L.sLastLvl = o; o += round4(L.Bp);
  L.sAdj = o; o += round4(2 * L.Pp);
  L.sPb = o; o += round4((L.Pp + 3) / 4);
  L.sPt = o; o += round4((L.Pp + 3) / 4);
  L.sPr = o; o += round4(L.Pp);
  L.sBk = o; o += round4((L.Bp + 3) / 4);
  L.sDamp = o; o += round4(2 * L.Bp);
  L.sLc = o; o += round4(LC_WORDS * std::max((int)s0.num_lights, 1));
  L.sBmask = o; o += round4(L.Bp * L.KW);
  L.sEnt = o; o += L.Kmax;
  L.sEntC = o; o += round4((L.Kmax + 1) / 2);
  L.sGs = o; o += round4((L.Kmax + 3) / 4);
  // the touching list, the constraint order and the level table are dead once the schedule (ent/entC) is built,
  // which is before the first constraint record is written: they share the records' space
  L.sRec = o;
  L.sTl = o;
  L.sOrd = o + L.Kmax;
  L.sLvlTab = o + 2 * L.Kmax;
  // (outside solve() the region also holds the TOI alpha cache at 3*Kmax+8 and, after it, general records)
  L.recWords = round4(std::max(std::max(std::max(8 * L.Kmax, 2 * L.Kmax + round4(L.Kmax + 2)), 2 * L.Pp),
                               3 * L.Kmax + 8 + L.Cmax + 2 * GR_WORDS));
  o += L.recWords;
  L.sMisc = o; o += 8;
  L.smemWords = round4(o);
  }
  L.stepsPerAction = s0.steps_per_action;
  L.velIters = s0.velocity_iterations;
  L.posIters = s0.position_iterations;
  L.dampingMode = s0.damping_mode;
  L.enableToi = s0.enable_toi;
  L.enableSleep = s0.enable_sleep;
  L.dt = s0.dt;
  {
    // Kilobot.step single-motor branches, lib/kilobot.py:103-121 (float64, then b2Vec2 float32)
    const double legLeft[2] = {-0.013, -0.009}, legRight[2] = {+0.013, -0.009};
    const double maxAngular = 0.5 * M_PI, dt = 1. / 10;
    double av = 255 / 255. * maxAngular, ad = av * dt;
    double c = std::cos(ad), s = std::sin(ad);
    L.transRight[0] = (float)((legLeft[0] - (c * legLeft[0] + (-s) * legLeft[1])) * 25.0);
    L.transRight[1] = (float)((legLeft[1] - (s * legLeft[0] + c * legLeft[1])) * 25.0);
    L.omegaRight = (float)av;
    av = -255 / 255. * maxAngular;
    ad = av * dt;
    c = std::cos(ad);
    s = std::sin(ad);
    L.transLeft[0] = (float)((legRight[0] - (c * legRight[0] + (-s) * legRight[1])) * 25.0);
    L.transLeft[1] = (float)((legRight[1] - (s * legRight[0] + c * legRight[1])) * 25.0);
    L.omegaLeft = (float)av;
  }
  if (swarm) {
    h->envsPerBlock = 1;
    h->smemBytes = (size_t)h->W.smemBytes;
  } else {
    int lpe = B <= 6 ? 4 : (B <= 24 ? 8 : (B <= 40 ? 16 : 32));
    if (const char* ev = getenv("KB_LANES_PER_ENV")) {
      const int v = atoi(ev);
      if (v == 4 || v == 8 || v == 16 || v == 32) lpe = v;
    }
    L.lanesPerEnv = lpe;
#ifndef KB_NO_BANK_STAGGER
    // stagger the lane groups of a warp over the 32 shared-memory banks: with a per-env stride of LPE (mod 32) words
    // the groups' copies of the same field start LPE banks apart, so a word access by every lane of the warp is one
    // wavefront instead of up to 32 / LPE (a stride of 0 mod 32 cost 30 % extra wavefronts, profiles/)
    if (lpe < 32)
      while (L.smemWords % 32 != lpe) L.smemWords += 4;
#endif
    h->envsPerBlock = KB_BLOCK_OF(L.lanesPerEnv) / L.lanesPerEnv;
    h->smemBytes = (size_t)h->envsPerBlock * L.smemWords * 4;
  }
  return KB_OK;
}

}  // namespace kb

using namespace kb;

extern "C" {

const char* kb_last_error(void) { return g_err.c_str(); }

int kb_create(const KbSceneDesc* scenes, int32_t num_scenes, const int32_t* env_scene, int32_t num_envs,
              int32_t max_contacts, int32_t device, KbHandle** out) {
  if (!scenes || num_scenes < 1 || num_envs < 1 || !out) return fail(KB_ERR_INVALID, "kb_create: invalid arguments");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
    cudaGetLastError();
    return fail(KB_ERR_NO_DEVICE, "kb_create: no CUDA device (this library has no CPU fallback)");
  }
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(KB_ERR_NO_DEVICE, "kb_create: device is not sm_100 (B200); no fallback path exists");
  CUDA_TRY(cudaSetDevice(device));

  Handle* h = new Handle();
  h->device = device;
  h->numEnvs = num_envs;
  h->numScenes = num_scenes;
  {
    const int rc = planBatch(scenes, num_scenes, max_contacts, prop, h);
    if (rc != KB_OK) {
      delete h;
      return rc;
    }
  }
  const KbSceneDesc& s0 = scenes[0];
  const Layout& L = h->L;
  const bool swarm = h->W.enabled != 0;
  const int M = L.M, N = L.N;
  if (h->smemBytes > (size_t)prop.sharedMemPerBlockOptin) {
    delete h;
    return fail(KB_ERR_CAPACITY, swarm ? "kb_create: this swarm does not fit one SM's shared memory (about 1700 kilobots per env at the minimal capacities)"
                                       : "kb_create: per-env shared-memory image too large; lower max_contacts");
  }

  std::vector<ProxyConst> allProxies;
  std::vector<BodyConst> allBodies;
  std::vector<SceneConst> allScenes(num_scenes);
  h->hostBodies.resize(num_scenes);
  for (int s = 0; s < num_scenes; ++s) {
    std::vector<ProxyConst> px;
    int rc = buildScene(scenes[s], L.M, L.Bp, L.Pp, &px, &h->hostBodies[s], &allScenes[s]);
    if (rc != KB_OK) {
      delete h;
      return rc;
    }
    allProxies.insert(allProxies.end(), px.begin(), px.end());
    h->hostNumProxies.push_back(allScenes[s].numProxies);
    h->hostNumObjects.push_back(scenes[s].num_objects);
    h->hostNumKilobots.push_back(scenes[s].num_bodies - scenes[s].num_objects);
    allBodies.insert(allBodies.end(), h->hostBodies[s].begin(), h->hostBodies[s].end());
  }
  const int NLp = std::max(1, (int)s0.num_lights);
  std::vector<LightConst> lights((size_t)NLp * num_scenes);   // [scene][light]
  std::memset(lights.data(), 0, sizeof(LightConst) * lights.size());
  for (int s = 0; s < num_scenes; ++s)
    for (int l = 0; l < s0.num_lights; ++l) {
      const KbLightDef& ld = scenes[s].lights[l];
      LightConst& lc = lights[(size_t)s * NLp + l];
      lc.type = ld.type;
      lc.relative = ld.relative_actions;
      lc.radius = ld.radius;
      for (int k = 0; k < 2; ++k) {
        lc.blo[k] = ld.bounds_lo[k];
        lc.bhi[k] = ld.bounds_hi[k];
        lc.alo[k] = ld.action_lo[k];
        lc.ahi[k] = ld.action_hi[k];
      }
      lc.maxVel = ld.max_velocity;
    }
#define ALLOC_COPY(dst, vec)                                                                   \
  CUDA_TRY(cudaMalloc(&(dst), sizeof((vec)[0]) * (vec).size()));                               \
  CUDA_TRY(cudaMemcpy((dst), (vec).data(), sizeof((vec)[0]) * (vec).size(), cudaMemcpyHostToDevice));
  ALLOC_COPY(h->dProxies, allProxies);
  ALLOC_COPY(h->dBodies, allBodies);
  ALLOC_COPY(h->dScenes, allScenes);
  ALLOC_COPY(h->dLights, lights);
#undef ALLOC_COPY
  if (env_scene) {
    for (int i = 0; i < num_envs; ++i)
      if (env_scene[i] < 0 || env_scene[i] >= num_scenes) return fail(KB_ERR_INVALID, "kb_create: env_scene out of range");
    CUDA_TRY(cudaMalloc(&h->dEnvScene, sizeof(int32_t) * num_envs));
    CUDA_TRY(cudaMemcpy(h->dEnvScene, env_scene, sizeof(int32_t) * num_envs, cudaMemcpyHostToDevice));
  }
  const size_t blobBytes = (size_t)launchGrid(h) * h->envsPerBlock * L.blobWords * 4;  // padded to whole blocks
  CUDA_TRY(cudaMalloc(&h->dBlobs, blobBytes));
  CUDA_TRY(cudaMemset(h->dBlobs, 0, blobBytes));
  if (env_scene)   // H_SCENE before the first reset: the env's scene, so that kb_get_body_counts is right from the start
    CUDA_TRY(cudaMemcpy2D(h->dBlobs + L.oHdr + H_SCENE, (size_t)L.blobWords * 4, env_scene, sizeof(int32_t), sizeof(int32_t),
                          (size_t)num_envs, cudaMemcpyHostToDevice));
  const int Amax = std::max(std::max(L.A, 2 * N), 1);
  CUDA_TRY(cudaMalloc(&h->dAction, sizeof(double) * (size_t)num_envs * Amax));
  {
    const int64_t sizes[6] = {(int64_t)sizeof(float) * num_envs * N * 3, (int64_t)sizeof(float) * num_envs * M * 3,
                              (int64_t)sizeof(double) * num_envs * L.L, (int64_t)sizeof(float) * num_envs,
                              (int64_t)sizeof(int32_t) * num_envs, (int64_t)num_envs};
    int64_t off = 0;
    for (int i = 0; i < 6; ++i) {
      h->hostOff[i] = off;
      off += (sizes[i] + 255) & ~(int64_t)255;
    }
    h->hostTotal = off;
    CUDA_TRY(cudaMalloc(&h->dOut, (size_t)off + 256));
    h->dObsK = reinterpret_cast<float*>(h->dOut + h->hostOff[0]);
    h->dObsO = reinterpret_cast<float*>(h->dOut + h->hostOff[1]);
    h->dObsL = reinterpret_cast<double*>(h->dOut + h->hostOff[2]);
    h->dReward = reinterpret_cast<float*>(h->dOut + h->hostOff[3]);
    h->dStatus = reinterpret_cast<int32_t*>(h->dOut + h->hostOff[4]);
    h->dDone = h->dOut + h->hostOff[5];
  }
  h->wall[0] = s0.wall_x0; h->wall[1] = s0.wall_y0; h->wall[2] = s0.wall_x1; h->wall[3] = s0.wall_y1;
  CUDA_TRY(cudaMalloc(&h->dTask, sizeof(double) * KB_TASK_WORDS * (size_t)num_envs));
  CUDA_TRY(cudaMemset(h->dTask, 0, sizeof(double) * KB_TASK_WORDS * (size_t)num_envs));
#ifdef KB_PROFILE
  CUDA_TRY(cudaMalloc(&h->dProf, sizeof(unsigned long long) * KB_PROF_SLOTS * (size_t)num_envs));
#endif
#define KB_SET_SMEM(LPE)                                                                                            \
  case LPE:                                                                                                          \
    CUDA_TRY(raiseSmemLimit(kb_step_kernel<LPE>, h->smemBytes));                                                     \
    CUDA_TRY(raiseSmemLimit(kb_reset_kernel<LPE>, h->smemBytes));                                                    \
    CUDA_TRY(raiseSmemLimit(kb_setpose_kernel<LPE>, h->smemBytes));                                                  \
    break;
  if (swarm) {
#define KB_SET_SWARM_SMEM(T)                                                                                           \
    CUDA_TRY(raiseSmemLimit(kb_swarm_step_kernel<T>, h->smemBytes));                                                 \
    CUDA_TRY(raiseSmemLimit(kb_swarm_reset_kernel<T>, h->smemBytes));                                                \
    CUDA_TRY(raiseSmemLimit(kb_swarm_setpose_kernel<T>, h->smemBytes));
    if (L.lanesPerEnv == 128) { KB_SET_SWARM_SMEM(128) } else if (L.lanesPerEnv == 256) { KB_SET_SWARM_SMEM(256) } else { KB_SET_SWARM_SMEM(512) }
#undef KB_SET_SWARM_SMEM
  } else switch (L.lanesPerEnv) {
    KB_SET_SMEM(4)
    KB_SET_SMEM(8)
    KB_SET_SMEM(16)
    KB_SET_SMEM(32)
  }
#undef KB_SET_SMEM
  if (!swarm) {
    // KB_JIT=0: the generic kernel; KB_JIT=1: the specialised kernel or an error; unset: the specialised kernel when
    // it can be had
    const char* ev = getenv("KB_JIT");
    const int mode = ev && *ev ? atoi(ev) : -1;
    if (mode == 0) {
      h->jitReason = "KB_JIT=0";
    } else {
      double ms = 0.0;
      h->stepJit = jitStepKernel(L, &ms, &h->jitReason);
      h->jitMs = (float)ms;
      if (h->stepJit) {
        const cudaError_t e = raiseSmemLimit((const void*)h->stepJit, h->smemBytes);
        if (e != cudaSuccess) {
          cudaGetLastError();
          h->stepJit = nullptr;
          h->jitReason = std::string("load error: ") + cudaGetErrorString(e);
        }
      }
      if (!h->stepJit && mode == 1) {
        const std::string why = h->jitReason;
        kb_destroy(reinterpret_cast<KbHandle*>(h));
        return fail(KB_ERR_CUDA, "kb_create: KB_JIT=1 but the specialised step kernel is not available: " + why);
      }
    }
  } else {
    h->jitReason = "large-swarm tier";
  }
  {
    // end-to-end pipeline depth: one chunk per ~2 MB of outputs, at most 8, each a whole number of blocks and at
    // least a few waves long (small batches -- C2's 4096 envs are ONE wave -- stay a single launch)
    const int64_t chunkBytes = 2 << 20;
    int nc = (int)std::min<int64_t>(8, std::max<int64_t>(1, h->hostTotal / chunkBytes));
    const int blocks = launchGrid(h);
    while (nc > 1 && blocks / nc < 4 * 148) --nc;
    if (const char* ev = getenv("KB_HOST_CHUNKS")) nc = std::max(1, std::min(64, atoi(ev)));
    h->hostChunks = nc;
    if (nc > 1) {
      for (int i = 0; i < 2; ++i) {
        CUDA_TRY(cudaStreamCreateWithFlags(&h->pipe[i], cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&h->evJoin[i], cudaEventDisableTiming));
      }
      CUDA_TRY(cudaEventCreateWithFlags(&h->evFork, cudaEventDisableTiming));
    }
  }
  *out = reinterpret_cast<KbHandle*>(h);
  return KB_OK;
}

int kb_destroy(KbHandle* hh) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return KB_OK;
  cudaSetDevice(h->device);
  cudaFree(h->dBlobs); cudaFree(h->dEnvScene); cudaFree(h->dProxies); cudaFree(h->dBodies);
  cudaFree(h->dScenes); cudaFree(h->dLights); cudaFree(h->dAction); cudaFree(h->dOut); cudaFree(h->dTask); cudaFree(h->dRenderIds);
  cudaFree(h->dSampler); cudaFree(h->dSamplePose); cudaFree(h->dSampleLight); cudaFree(h->dEpisode);
  cudaFree(h->dSceneConfig); cudaFree(h->dConfigCdf);
  for (int i = 0; i < 2; ++i) {
    if (h->pipe[i]) cudaStreamDestroy(h->pipe[i]);
    if (h->evJoin[i]) cudaEventDestroy(h->evJoin[i]);
  }
  if (h->evFork) cudaEventDestroy(h->evFork);
  delete h;
  return KB_OK;
}

int kb_get_dims(const KbHandle* hh, KbDims* d) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h || !d) return fail(KB_ERR_INVALID, "kb_get_dims: null");
  d->num_envs = h->numEnvs;
  d->num_bodies = h->L.B;
  d->num_objects = h->L.M;
  d->num_kilobots = h->L.N;
  d->num_proxies = h->L.P;
  d->max_contacts = h->L.Cmax;
  d->light_state_dim = h->L.L;
  d->action_dim = h->L.A;
  d->state_bytes_per_env = h->L.blobWords * 4;
  return KB_OK;
}

// launches `kernel` over the envs [a.envOffset, a.envOffset + count)
#define KB_LAUNCH_RANGE(kernel, swarmKernel, h, st, a, count)                                     \
  if ((h)->W.enabled) {                                                                           \
    switch ((h)->L.lanesPerEnv) {                                                                 \
      case 128: swarmKernel<128><<<(count), 128, (h)->smemBytes, (st)>>>(a); break;                     \
      case 256: swarmKernel<256><<<(count), 256, (h)->smemBytes, (st)>>>(a); break;                     \
      default: swarmKernel<512><<<(count), 512, (h)->smemBytes, (st)>>>(a); break;                      \
    }                                                                                             \
  } else {                                                                                        \
    const int grid_ = ((count) + (h)->envsPerBlock - 1) / (h)->envsPerBlock;                      \
    switch ((h)->L.lanesPerEnv) {                                                                 \
      case 4: kernel<4><<<grid_, KB_BLOCK_OF(4), (h)->smemBytes, (st)>>>(a); break;                     \
      case 8: kernel<8><<<grid_, KB_BLOCK_OF(8), (h)->smemBytes, (st)>>>(a); break;                     \
      case 16: kernel<16><<<grid_, KB_BLOCK_OF(16), (h)->smemBytes, (st)>>>(a); break;                   \
      default: kernel<32><<<grid_, KB_BLOCK_OF(32), (h)->smemBytes, (st)>>>(a); break;                   \
    }                                                                                             \
  }
#define KB_LAUNCH(kernel, swarmKernel, h, st, a) KB_LAUNCH_RANGE(kernel, swarmKernel, h, st, a, (h)->numEnvs)

int kb_reset(KbHandle* hh, const uint8_t* mask, const double* body_pose, const double* light_state,
             const double* kb_velocity, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !body_pose) return fail(KB_ERR_INVALID, "kb_reset: null handle or poses");
  if (h->L.L > 0 && !light_state) return fail(KB_ERR_INVALID, "kb_reset: light_state required");
  CUDA_TRY(cudaSetDevice(h->device));
  KernelArgs a;
  fillArgs(h, &a);
  a.mask = mask;
  a.pose = body_pose;
  a.lightInit = light_state;
  a.kbVel = kb_velocity;
  a.status = h->dStatus;
  KB_LAUNCH(kb_reset_kernel, kb_swarm_reset_kernel, h, (cudaStream_t)stream, a);
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

// ---- on-device scene sampling (include/kb_b200.h "Reset with on-device scene sampling") ------------------------
}  // extern "C"

namespace kb {
// Validates K sampler specs against the batch and uploads them (kb_set_sampler is the case K = 1): the configurations,
// the configuration of every scene and the normalised cumulative weights (weights == NULL: the env's scene decides).
static int setSamplers(Handle* h, const KbSampleSpec* specs, int K, const double* weights, const char* who) {
  const Layout& L = h->L;
  auto bad = [&](const char* what) { return fail(KB_ERR_INVALID, std::string(who) + ": " + what); };
  if (K < 1 || K > KB_SAMPLE_MAX_CONFIGS) return bad("num_specs must be 1..16");
  std::vector<int> sceneConfig(h->numScenes, -1);
  std::vector<SamplerConst> scs(K);
  for (int c = 0; c < K; ++c) {
    const KbSampleSpec* spec = specs + c;
    if (spec->seed != specs[0].seed || spec->env_id_base != specs[0].env_id_base)
      return bad("seed and env_id_base must be equal over the specs");
    if (spec->num_objects < 0 || spec->num_objects > KB_SAMPLE_MAX_OBJECTS) return bad("num_objects must be at most 16");
    if (spec->num_lights != L.numLights) return bad("num_lights must equal the batch's");
    if ((spec->num_objects > 0 && !spec->objects) || (spec->num_lights > 0 && !spec->lights))
      return bad("missing object / light descriptions");
    const bool shuffle = spec->shuffle_lights && spec->num_lights > 1;
    // the scenes of this configuration: one per permutation of a shuffled light, else its one scene; with K = 1 and no
    // shuffle every scene of the batch (the env keeps its scene)
    std::vector<int> mine;
    int nperm = 1;
    if (shuffle)
      for (int q = 2; q <= spec->num_lights; ++q) nperm *= q;
    if (shuffle || K > 1) {
      if (!spec->perm_scene) return bad(shuffle ? "shuffle_lights needs perm_scene" : "perm_scene is required with more than one spec");
      for (int r = 0; r < nperm; ++r) {
        if (spec->perm_scene[r] < 0 || spec->perm_scene[r] >= h->numScenes) return bad("perm_scene out of range");
        mine.push_back(spec->perm_scene[r]);
      }
    } else {
      for (int sc = 0; sc < h->numScenes; ++sc) mine.push_back(sc);
    }
    for (int s : mine) {
      if (h->hostNumObjects[s] != spec->num_objects) return bad("num_objects must equal the object count of each of the spec's scenes");
      if (h->hostNumKilobots[s] != h->hostNumKilobots[mine[0]]) return bad("the scenes of a spec must have one kilobot count");
      if (sceneConfig[s] >= 0 && sceneConfig[s] != c) return bad("a scene belongs to two specs");
      sceneConfig[s] = c;
    }
    SamplerConst& sc = scs[c];
    std::memset(&sc, 0, sizeof(sc));
    sc.seedLo = (uint32_t)(spec->seed & 0xFFFFFFFFull);
    sc.seedHi = (uint32_t)(spec->seed >> 32);
    sc.envIdBase = spec->env_id_base;
    sc.sizeX = spec->world_width;
    sc.sizeY = spec->world_height;
    sc.numObjects = spec->num_objects;
    sc.numLights = spec->num_lights;
    sc.meanMode = spec->kilobot_mean_mode;
    sc.mean[0] = spec->kilobot_mean[0];
    sc.mean[1] = spec->kilobot_mean[1];
    sc.std = spec->kilobot_std;
    for (int i = 0; i < spec->num_objects; ++i) {
      sc.objMode[i] = spec->objects[i].mode;
      for (int k = 0; k < 3; ++k) sc.objPose[i][k] = spec->objects[i].pose[k];
      sc.objExtent[i] = spec->objects[i].extent;
    }
    for (int l = 0; l < spec->num_lights; ++l) {
      sc.lightMode[l] = spec->lights[l].mode;
      if (sc.lightMode[l] == KB_SAMPLE_AT_OBJECT && spec->num_objects == 0) return bad("light init 'object' without objects");
      sc.lightInit[l][0] = spec->lights[l].init[0];
      sc.lightInit[l][1] = spec->lights[l].init[1];
    }
    sc.shuffle = shuffle;
    if (shuffle || K > 1)
      for (int r = 0; r < nperm; ++r) sc.permScene[r] = spec->perm_scene[r];
    sc.ownScene = !shuffle && K > 1;
  }
  std::vector<double> cdf(KB_SAMPLE_MAX_CONFIGS, 1.0);
  if (weights) {
    double total = 0.0;
    for (int c = 0; c < K; ++c) {
      if (!std::isfinite(weights[c]) || weights[c] < 0.0) return bad("weights must be finite and non-negative");
      total += weights[c];
    }
    if (!(total > 0.0) || !std::isfinite(total)) return bad("weights must have a positive (finite) sum");
    // from the last configuration of positive weight on, exactly 1.0: u < 1 always finds one, never a zero weight
    int last = K - 1;
    while (weights[last] == 0.0) --last;
    double acc = 0.0;
    for (int c = 0; c < K; ++c) {
      acc += weights[c];
      cdf[c] = c >= last ? 1.0 : acc / total;
    }
  }
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  const size_t E = (size_t)h->numEnvs;
  std::vector<int32_t> envScene(E, 0);
  if (h->dEnvScene) CUDA_TRY(cudaMemcpy(envScene.data(), h->dEnvScene, sizeof(int32_t) * E, cudaMemcpyDeviceToHost));
  if (K > 1)
    for (size_t e = 0; e < E; ++e)
      if (sceneConfig[envScene[e]] < 0) return bad("an env's scene belongs to no spec");
  if (!h->dSampler) {
    CUDA_TRY(cudaMalloc(&h->dSampler, sizeof(SamplerConst) * KB_SAMPLE_MAX_CONFIGS));
    CUDA_TRY(cudaMalloc(&h->dSamplePose, sizeof(double) * E * L.B * 3));
    CUDA_TRY(cudaMalloc(&h->dSampleLight, sizeof(double) * E * std::max(L.L, 1)));
    CUDA_TRY(cudaMalloc(&h->dEpisode, sizeof(uint32_t) * E));
    CUDA_TRY(cudaMalloc(&h->dSceneConfig, sizeof(int32_t) * h->numScenes));
    CUDA_TRY(cudaMalloc(&h->dConfigCdf, sizeof(double) * KB_SAMPLE_MAX_CONFIGS));
  }
  CUDA_TRY(cudaMemset(h->dEpisode, 0, sizeof(uint32_t) * E));
  CUDA_TRY(cudaMemcpy(h->dSampler, scs.data(), sizeof(SamplerConst) * K, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->dSceneConfig, sceneConfig.data(), sizeof(int32_t) * h->numScenes, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->dConfigCdf, cdf.data(), sizeof(double) * KB_SAMPLE_MAX_CONFIGS, cudaMemcpyHostToDevice));
  if (!h->dEnvScene) {   // the reset may switch scenes: the per-env scene map becomes device state
    CUDA_TRY(cudaMalloc(&h->dEnvScene, sizeof(int32_t) * E));
    CUDA_TRY(cudaMemset(h->dEnvScene, 0, sizeof(int32_t) * E));
  }
  h->numConfigs = K;
  h->weighted = weights != nullptr;
  h->hostSceneConfig = sceneConfig;
  return KB_OK;
}
}  // namespace kb

extern "C" {

int kb_set_sampler(KbHandle* hh, const KbSampleSpec* spec) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !spec) return fail(KB_ERR_INVALID, "kb_set_sampler: null");
  for (int s = 0; s < h->numScenes; ++s)
    if (h->hostNumObjects[s] != h->L.M || h->hostNumKilobots[s] != h->L.N)
      return fail(KB_ERR_UNSUPPORTED, "kb_set_sampler: the scenes differ in their object / kilobot counts (draw them with kb_set_sampler_mix)");
  return setSamplers(h, spec, 1, nullptr, "kb_set_sampler");
}

int kb_set_sampler_mix(KbHandle* hh, const KbSampleSpec* specs, int32_t num_specs, const double* weights) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !specs) return fail(KB_ERR_INVALID, "kb_set_sampler_mix: null");
  return setSamplers(h, specs, num_specs, weights, "kb_set_sampler_mix");
}

int kb_current_scenes(KbHandle* hh, int32_t* out_device, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !out_device) return fail(KB_ERR_INVALID, "kb_current_scenes: null");
  CUDA_TRY(cudaSetDevice(h->device));
  kb_current_scenes_kernel<<<(h->numEnvs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->dBlobs, h->L.blobWords,
                                                                                      h->L.oHdr + H_SCENE, h->numEnvs, out_device);
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

int kb_reset_sampled(KbHandle* hh, const uint8_t* mask, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return fail(KB_ERR_INVALID, "kb_reset_sampled: null handle");
  if (!h->dSampler) return fail(KB_ERR_INVALID, "kb_reset_sampled: no sampler (kb_set_sampler)");
  CUDA_TRY(cudaSetDevice(h->device));
  KernelArgs a;
  fillArgs(h, &a);
  a.mask = mask;
  a.pose = h->dSamplePose;
  a.lightInit = h->dSampleLight;
  a.kbVel = nullptr;
  a.status = h->dStatus;
  a.sampler = h->dSampler;
  a.samplePose = h->dSamplePose;
  a.sampleLight = h->dSampleLight;
  a.envSceneW = h->dEnvScene;
  a.episode = h->dEpisode;
  a.sceneConfig = h->dSceneConfig;
  a.configCdf = h->weighted ? h->dConfigCdf : nullptr;
  a.numConfigs = h->numConfigs;
  KB_LAUNCH(kb_reset_kernel, kb_swarm_reset_kernel, h, (cudaStream_t)stream, a);
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

int kb_get_sampled(KbHandle* hh, double* body_pose, double* light_state, int32_t* env_scene, uint32_t* episodes) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !h->dSampler) return fail(KB_ERR_INVALID, "kb_get_sampled: no sampler");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  const size_t E = (size_t)h->numEnvs;
  if (body_pose) CUDA_TRY(cudaMemcpy(body_pose, h->dSamplePose, sizeof(double) * E * h->L.B * 3, cudaMemcpyDeviceToHost));
  if (light_state && h->L.L > 0) CUDA_TRY(cudaMemcpy(light_state, h->dSampleLight, sizeof(double) * E * h->L.L, cudaMemcpyDeviceToHost));
  if (env_scene) CUDA_TRY(cudaMemcpy(env_scene, h->dEnvScene, sizeof(int32_t) * E, cudaMemcpyDeviceToHost));
  if (episodes) CUDA_TRY(cudaMemcpy(episodes, h->dEpisode, sizeof(uint32_t) * E, cudaMemcpyDeviceToHost));
  return KB_OK;
}

int kb_set_env_scene(KbHandle* hh, const int32_t* env_scene) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !env_scene) return fail(KB_ERR_INVALID, "kb_set_env_scene: null");
  for (int i = 0; i < h->numEnvs; ++i)
    if (env_scene[i] < 0 || env_scene[i] >= h->numScenes) return fail(KB_ERR_INVALID, "kb_set_env_scene: scene out of range");
    else if (h->numConfigs > 1 && h->hostSceneConfig[env_scene[i]] < 0)
      return fail(KB_ERR_INVALID, "kb_set_env_scene: the scene belongs to no configuration of the sampler");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  if (!h->dEnvScene) CUDA_TRY(cudaMalloc(&h->dEnvScene, sizeof(int32_t) * (size_t)h->numEnvs));
  CUDA_TRY(cudaMemcpy(h->dEnvScene, env_scene, sizeof(int32_t) * (size_t)h->numEnvs, cudaMemcpyHostToDevice));
  return KB_OK;
}

static int stepRange(Handle* h, const double* action, int32_t action_mode, float* obs_kilobots, float* obs_objects,
                     double* obs_light, float* reward, uint8_t* done, int32_t* status, int envBegin, int envCount,
                     cudaStream_t stream) {
  KernelArgs a;
  fillArgs(h, &a);
  a.action = action_mode == KB_ACTION_NONE ? nullptr : action;
  a.actionMode = a.action || action_mode == KB_ACTION_KILOBOTS ? action_mode : KB_ACTION_NONE;
  a.obsKilobots = obs_kilobots;
  a.obsObjects = obs_objects;
  a.obsLight = obs_light;
  a.reward = reward;
  a.done = done;
  a.status = status;
  a.obsFlat = h->obsFlat;
  a.envOffset = envBegin;
  if (h->stepJit) {
    void* args[] = {&a};
    const int grid = (envCount + h->envsPerBlock - 1) / h->envsPerBlock;
    CUDA_TRY(cudaLaunchKernel((const void*)h->stepJit, dim3(grid), dim3(KB_BLOCK_OF(h->L.lanesPerEnv)), args,
                              h->smemBytes, stream));
    return KB_OK;
  }
  KB_LAUNCH_RANGE(kb_step_kernel, kb_swarm_step_kernel, h, stream, a, envCount);
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

int kb_step(KbHandle* hh, const double* action, int32_t action_mode, float* obs_kilobots, float* obs_objects,
            double* obs_light, float* reward, uint8_t* done, int32_t* status, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return fail(KB_ERR_INVALID, "kb_step: null handle");
  if (action_mode != KB_ACTION_NONE && action_mode != KB_ACTION_LIGHT && action_mode != KB_ACTION_KILOBOTS)
    return fail(KB_ERR_INVALID, "kb_step: bad action_mode");
  CUDA_TRY(cudaSetDevice(h->device));
  return stepRange(h, action, action_mode, obs_kilobots, obs_objects, obs_light, reward, done, status, 0, h->numEnvs,
                   (cudaStream_t)stream);
}

int kb_step_host(KbHandle* hh, const double* action, int32_t action_mode, float* obs_kilobots, float* obs_objects,
                 double* obs_light, float* reward, uint8_t* done, int32_t* status, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return fail(KB_ERR_INVALID, "kb_step_host: null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const Layout& L = h->L;
  const size_t E = (size_t)h->numEnvs;
  if (action_mode != KB_ACTION_NONE && action_mode != KB_ACTION_LIGHT && action_mode != KB_ACTION_KILOBOTS)
    return fail(KB_ERR_INVALID, "kb_step_host: bad action_mode");
  if (h->hostChunks > 1) {
    // pipelined: chunk c = H2D of its actions, kernel over its envs, D2H of its outputs, on side stream c % 2; the
    // copies of one chunk overlap the kernel of the next.  Chunks are whole blocks; only the last one is ragged.
    const size_t A = action_mode == KB_ACTION_KILOBOTS ? 2 * (size_t)L.N : (size_t)L.A;
    const bool haveAct = action && action_mode != KB_ACTION_NONE;
    const int epb = h->envsPerBlock, blocks = launchGrid(h), nc = h->hostChunks;
    CUDA_TRY(cudaEventRecord(h->evFork, st));
    for (int i = 0; i < 2; ++i) CUDA_TRY(cudaStreamWaitEvent(h->pipe[i], h->evFork, 0));
    for (int c = 0; c < nc; ++c) {
      const int b0 = (int)((int64_t)blocks * c / nc), b1 = (int)((int64_t)blocks * (c + 1) / nc);
      const int e0 = b0 * epb, e1 = std::min(b1 * epb, h->numEnvs);
      if (e1 <= e0) continue;
      const size_t n = (size_t)(e1 - e0);
      cudaStream_t s = h->pipe[c & 1];
      if (haveAct) CUDA_TRY(cudaMemcpyAsync(h->dAction + (size_t)e0 * A, action + (size_t)e0 * A, sizeof(double) * n * A, cudaMemcpyHostToDevice, s));
      int rc = stepRange(h, haveAct ? h->dAction : nullptr, action_mode, obs_kilobots ? h->dObsK : nullptr,
                         obs_objects ? h->dObsO : nullptr, obs_light ? h->dObsL : nullptr, reward ? h->dReward : nullptr,
                         done ? h->dDone : nullptr, status ? h->dStatus : nullptr, e0, e1 - e0, s);
      if (rc != KB_OK) return rc;
      if (obs_kilobots && L.N > 0) CUDA_TRY(cudaMemcpyAsync(obs_kilobots + (size_t)e0 * L.N * 3, h->dObsK + (size_t)e0 * L.N * 3, sizeof(float) * n * L.N * 3, cudaMemcpyDeviceToHost, s));
      if (obs_objects && L.M > 0) CUDA_TRY(cudaMemcpyAsync(obs_objects + (size_t)e0 * L.M * 3, h->dObsO + (size_t)e0 * L.M * 3, sizeof(float) * n * L.M * 3, cudaMemcpyDeviceToHost, s));
      if (obs_light && L.L > 0) CUDA_TRY(cudaMemcpyAsync(obs_light + (size_t)e0 * L.L, h->dObsL + (size_t)e0 * L.L, sizeof(double) * n * L.L, cudaMemcpyDeviceToHost, s));
      if (reward) CUDA_TRY(cudaMemcpyAsync(reward + e0, h->dReward + e0, sizeof(float) * n, cudaMemcpyDeviceToHost, s));
      if (done) CUDA_TRY(cudaMemcpyAsync(done + e0, h->dDone + e0, n, cudaMemcpyDeviceToHost, s));
      if (status) CUDA_TRY(cudaMemcpyAsync(status + e0, h->dStatus + e0, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s));
    }
    for (int i = 0; i < 2; ++i) {
      CUDA_TRY(cudaEventRecord(h->evJoin[i], h->pipe[i]));
      CUDA_TRY(cudaStreamWaitEvent(st, h->evJoin[i], 0));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return KB_OK;
  }
  const double* dAct = nullptr;
  if (action && action_mode != KB_ACTION_NONE) {
    const size_t A = action_mode == KB_ACTION_KILOBOTS ? 2 * (size_t)L.N : (size_t)L.A;
    CUDA_TRY(cudaMemcpyAsync(h->dAction, action, sizeof(double) * E * A, cudaMemcpyHostToDevice, st));
    dAct = h->dAction;
  }
  int rc = kb_step(hh, dAct, action_mode, obs_kilobots ? h->dObsK : nullptr, obs_objects ? h->dObsO : nullptr,
                   obs_light ? h->dObsL : nullptr, reward ? h->dReward : nullptr, done ? h->dDone : nullptr,
                   status ? h->dStatus : nullptr, stream);
  if (rc != KB_OK) return rc;
  {
    // one device->host copy when the caller's buffers are laid out like the staging area (kb_get_host_layout)
    const uint8_t* base = reinterpret_cast<const uint8_t*>(obs_kilobots);
    const bool packed = obs_kilobots && obs_objects && obs_light && reward && done && status &&
                        reinterpret_cast<const uint8_t*>(obs_objects) == base + h->hostOff[1] &&
                        reinterpret_cast<const uint8_t*>(obs_light) == base + h->hostOff[2] &&
                        reinterpret_cast<const uint8_t*>(reward) == base + h->hostOff[3] &&
                        reinterpret_cast<const uint8_t*>(status) == base + h->hostOff[4] &&
                        reinterpret_cast<const uint8_t*>(done) == base + h->hostOff[5];
    if (packed) {
      CUDA_TRY(cudaMemcpyAsync(obs_kilobots, h->dOut, (size_t)h->hostTotal, cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      return KB_OK;
    }
  }
  if (obs_kilobots) CUDA_TRY(cudaMemcpyAsync(obs_kilobots, h->dObsK, sizeof(float) * E * L.N * 3, cudaMemcpyDeviceToHost, st));
  if (obs_objects && L.M > 0) CUDA_TRY(cudaMemcpyAsync(obs_objects, h->dObsO, sizeof(float) * E * L.M * 3, cudaMemcpyDeviceToHost, st));
  if (obs_light && L.L > 0) CUDA_TRY(cudaMemcpyAsync(obs_light, h->dObsL, sizeof(double) * E * L.L, cudaMemcpyDeviceToHost, st));
  if (reward) CUDA_TRY(cudaMemcpyAsync(reward, h->dReward, sizeof(float) * E, cudaMemcpyDeviceToHost, st));
  if (done) CUDA_TRY(cudaMemcpyAsync(done, h->dDone, E, cudaMemcpyDeviceToHost, st));
  if (status) CUDA_TRY(cudaMemcpyAsync(status, h->dStatus, sizeof(int32_t) * E, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return KB_OK;
}

// ---- introspection (host pointers, synchronous) ------------------------------------------------
static int fetchBlobs(Handle* h, std::vector<uint32_t>* buf) {
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  buf->resize((size_t)h->numEnvs * h->L.blobWords);
  CUDA_TRY(cudaMemcpy(buf->data(), h->dBlobs, buf->size() * 4, cudaMemcpyDeviceToHost));
  return KB_OK;
}
static inline float asf(uint32_t u) {
  float f;
  std::memcpy(&f, &u, 4);
  return f;
}

int kb_get_bodies(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> buf;
  int rc = fetchBlobs(h, &buf);
  if (rc) return rc;
  const Layout& L = h->L;
  for (int e = 0; e < h->numEnvs; ++e) {
    const uint32_t* w = buf.data() + (size_t)e * L.blobWords;
    for (int b = 0; b < L.B; ++b) {
      float* o = out + ((size_t)e * L.B + b) * KB_BODY_STATE_FLOATS;
      const uint32_t* pos = w + L.oPos + 4 * b;
      const uint32_t* vel = w + L.oVel + 4 * b;
      const uint32_t* xf = w + L.oXf + 4 * b;
      o[0] = asf(pos[0]); o[1] = asf(pos[1]); o[2] = asf(pos[2]);
      o[3] = asf(vel[0]); o[4] = asf(vel[1]); o[5] = asf(vel[2]);
      o[6] = asf(pos[3]);
      o[7] = (vel[3] & BF_AWAKE) ? 1.0f : 0.0f;
      o[8] = asf(xf[0]); o[9] = asf(xf[1]); o[10] = asf(xf[2]); o[11] = asf(xf[3]);
    }
  }
  return KB_OK;
}

int kb_set_poses_masked(KbHandle* hh, const double* body_pose, const uint8_t* body_mask) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !body_pose) return fail(KB_ERR_INVALID, "kb_set_poses: null");
  CUDA_TRY(cudaSetDevice(h->device));
  double* d = nullptr;
  uint8_t* dm = nullptr;
  const size_t nb = (size_t)h->numEnvs * h->L.B;
  const size_t bytes = sizeof(double) * nb * 3;
  CUDA_TRY(cudaMalloc(&d, bytes + (body_mask ? nb : 0)));
  CUDA_TRY(cudaMemcpy(d, body_pose, bytes, cudaMemcpyHostToDevice));
  if (body_mask) {
    dm = reinterpret_cast<uint8_t*>(d) + bytes;
    CUDA_TRY(cudaMemcpy(dm, body_mask, nb, cudaMemcpyHostToDevice));
  }
  KernelArgs a;
  fillArgs(h, &a);
  a.pose = d;
  a.mask = dm;
  KB_LAUNCH(kb_setpose_kernel, kb_swarm_setpose_kernel, h, (cudaStream_t)0, a);
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(d);
  if (e != cudaSuccess) return fail(KB_ERR_CUDA, cudaGetErrorString(e));
  return KB_OK;
}

int kb_set_poses(KbHandle* hh, const double* body_pose) { return kb_set_poses_masked(hh, body_pose, nullptr); }

int kb_get_status(KbHandle* hh, int32_t* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !out) return fail(KB_ERR_INVALID, "kb_get_status: null");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  // header word H_STATUS of every blob: one strided copy
  CUDA_TRY(cudaMemcpy2D(out, sizeof(int32_t), h->dBlobs + h->L.oHdr + H_STATUS, (size_t)h->L.blobWords * 4, sizeof(int32_t),
                        (size_t)h->numEnvs, cudaMemcpyDeviceToHost));
  return KB_OK;
}

int kb_get_body_counts(KbHandle* hh, int32_t* objects, int32_t* kilobots) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return fail(KB_ERR_INVALID, "kb_get_body_counts: null");
  std::vector<int32_t> scene((size_t)h->numEnvs);
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  // header word H_SCENE of every blob: the scene each env was last reset with
  CUDA_TRY(cudaMemcpy2D(scene.data(), sizeof(int32_t), h->dBlobs + h->L.oHdr + H_SCENE, (size_t)h->L.blobWords * 4,
                        sizeof(int32_t), (size_t)h->numEnvs, cudaMemcpyDeviceToHost));
  for (int e = 0; e < h->numEnvs; ++e) {
    const int s = scene[e] >= 0 && scene[e] < h->numScenes ? scene[e] : 0;
    if (objects) objects[e] = h->hostNumObjects[s];
    if (kilobots) kilobots[e] = h->hostNumKilobots[s];
  }
  return KB_OK;
}

int kb_get_contacts(KbHandle* hh, int32_t* pairs, int32_t* count) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> buf;
  int rc = fetchBlobs(h, &buf);
  if (rc) return rc;
  const Layout& L = h->L;
  for (int e = 0; e < h->numEnvs; ++e) {
    const uint32_t* w = buf.data() + (size_t)e * L.blobWords;
    const int nC = (int)w[L.oHdr + H_NC];
    count[e] = nC;
    for (int k = 0; k < nC && k < L.Cmax; ++k) {
      const int i = nC - 1 - k;  // world-list order: newest first
      const uint32_t info = w[L.oCw + i];
      int32_t* o = pairs + ((size_t)e * L.Cmax + k) * 4;
      o[0] = h->W.enabled ? (int32_t)(w[h->W.oCpair + i] & 0xFFFFu) : (int32_t)CW_PA(info);
      o[1] = h->W.enabled ? (int32_t)(w[h->W.oCpair + i] >> 16) : (int32_t)CW_PB(info);
      o[2] = (info & CI_TOUCHING) ? 1 : 0;
      o[3] = (int32_t)((info & CI_PC_MASK) >> CI_PC_SHIFT);
    }
  }
  return KB_OK;
}

int kb_get_impulses(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> buf;
  int rc = fetchBlobs(h, &buf);
  if (rc) return rc;
  const Layout& L = h->L;
  for (int e = 0; e < h->numEnvs; ++e) {
    const uint32_t* w = buf.data() + (size_t)e * L.blobWords;
    const int nC = (int)w[L.oHdr + H_NC];
    for (int k = 0; k < nC && k < L.Cmax; ++k) {
      const int i = nC - 1 - k;
      const uint32_t info = w[L.oCw + i];
      const int pc = (int)((info & CI_PC_MASK) >> CI_PC_SHIFT);
      float* o = out + ((size_t)e * L.Cmax + k) * 4;
      if (h->W.enabled) {   // swarm tier: one frictionless point per contact
        o[0] = pc > 0 ? asf(w[L.oMan + SR_WORDS * i + SR_IMP]) : 0.0f;
        o[1] = o[2] = o[3] = 0.0f;
        continue;
      }
      const uint32_t* rec = w + L.oMan + MR_WORDS * i;
      o[0] = pc > 0 ? asf(rec[MR_P0N]) : 0.0f;
      o[1] = pc > 0 ? asf(rec[MR_P0T]) : 0.0f;
      o[2] = pc > 1 ? asf(rec[MR_P1N]) : 0.0f;
      o[3] = pc > 1 ? asf(rec[MR_P1T]) : 0.0f;
    }
  }
  return KB_OK;
}

int kb_get_counters(KbHandle* hh, uint64_t* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> buf;
  int rc = fetchBlobs(h, &buf);
  if (rc) return rc;
  const Layout& L = h->L;
  for (int e = 0; e < h->numEnvs; ++e) {
    const uint32_t* w = buf.data() + (size_t)e * L.blobWords;
    std::memcpy(out + (size_t)e * KB_NUM_COUNTERS, w + L.oCnt, sizeof(uint64_t) * KB_NUM_COUNTERS);
  }
  return KB_OK;
}

int kb_get_proxies(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> buf;
  int rc = fetchBlobs(h, &buf);
  if (rc) return rc;
  const Layout& L = h->L;
  for (int e = 0; e < h->numEnvs; ++e) {
    const uint32_t* w = buf.data() + (size_t)e * L.blobWords;
    const int np = h->hostNumProxies[w[L.oHdr + H_SCENE]];
    std::memset(out + (size_t)e * L.P * 4, 0, sizeof(float) * 4 * L.P);
    std::memcpy(out + (size_t)e * L.P * 4, w + L.oFat, sizeof(float) * 4 * np);
  }
  return KB_OK;
}

int kb_get_controllers(KbHandle* hh, double* ctrl, double* light) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  std::vector<uint32_t> buf;
  int rc = fetchBlobs(h, &buf);
  if (rc) return rc;
  const Layout& L = h->L;
  for (int e = 0; e < h->numEnvs; ++e) {
    const uint32_t* w = buf.data() + (size_t)e * L.blobWords;
    if (ctrl) std::memcpy(ctrl + (size_t)e * L.N * 4, w + L.oCtrl, sizeof(double) * 4 * L.N);
    if (light) std::memcpy(light + (size_t)e * L.L, w + L.oLight, sizeof(double) * L.L);
  }
  return KB_OK;
}

int kb_get_state(KbHandle* hh, void* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !out) return fail(KB_ERR_INVALID, "kb_get_state: null");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(out, h->dBlobs, (size_t)h->numEnvs * h->L.blobWords * 4, cudaMemcpyDeviceToHost));
  return KB_OK;
}

int kb_set_state(KbHandle* hh, const void* in) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !in) return fail(KB_ERR_INVALID, "kb_set_state: null");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(h->dBlobs, in, (size_t)h->numEnvs * h->L.blobWords * 4, cudaMemcpyHostToDevice));
  return KB_OK;
}

#ifdef KB_PROFILE
// debug builds only: cycles per phase of the last kb_step, u64[E][KB_PROF_SLOTS]
int kb_get_profile(KbHandle* hh, unsigned long long* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(out, h->dProf, sizeof(unsigned long long) * KB_PROF_SLOTS * (size_t)h->numEnvs, cudaMemcpyDeviceToHost));
  return KB_OK;
}
#endif

int kb_get_host_layout(const KbHandle* hh, int64_t* offsets, int64_t* total) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h || !offsets || !total) return fail(KB_ERR_INVALID, "kb_get_host_layout: null");
  for (int i = 0; i < 6; ++i) offsets[i] = h->hostOff[i];
  *total = h->hostTotal;
  return KB_OK;
}

int kb_jit_step_source(const KbSceneDesc* scenes, int32_t num_scenes, int32_t max_contacts, int32_t compile,
                       char* source, int64_t source_cap, char* log, int64_t log_cap, double* compile_ms) {
  if (!scenes || num_scenes < 1 || !source || source_cap < 1) return fail(KB_ERR_INVALID, "kb_jit_step_source: invalid arguments");
  cudaDeviceProp prop;
  std::memset(&prop, 0, sizeof(prop));   // sizes only the large-swarm tier's image, which has no specialised kernel
  Handle h;
  const int rc = planBatch(scenes, num_scenes, max_contacts, prop, &h);
  if (rc != KB_OK) return rc;
  if (h.W.enabled) return fail(KB_ERR_INVALID, "kb_jit_step_source: the large-swarm tier has no specialised step kernel");
  const std::string prelude = jitPrelude(h.L);
  std::snprintf(source, (size_t)source_cap, "%s", prelude.c_str());
  if (!compile) return KB_OK;
  std::vector<char> cubin;
  std::string text, err;
  const auto t0 = std::chrono::steady_clock::now();
  const bool ok = jitCompile(prelude, &cubin, &text, &err);
  if (compile_ms) *compile_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (log && log_cap > 0) std::snprintf(log, (size_t)log_cap, "%s", text.c_str());
  return ok ? KB_OK : fail(KB_ERR_CUDA, "kb_jit_step_source: " + err);
}

int kb_get_launch_config(const KbHandle* hh, KbLaunchConfig* cfg) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h || !cfg) return fail(KB_ERR_INVALID, "kb_get_launch_config: null");
  cfg->lanes_per_env = h->L.lanesPerEnv;
  cfg->block_threads = h->W.enabled ? h->L.lanesPerEnv : KB_BLOCK_OF(h->L.lanesPerEnv);
  cfg->grid_blocks = launchGrid(h);
  cfg->smem_bytes_per_block = (int32_t)h->smemBytes;
  cfg->state_words_per_env = h->L.stateWords;
  cfg->smem_words_per_env = h->L.smemWords;
  cfg->specialised = h->stepJit != nullptr;
  cfg->jit_ms = h->jitMs;
  std::snprintf(cfg->jit_reason, sizeof(cfg->jit_reason), "%s", h->jitReason.c_str());
  return KB_OK;
}

// ---- task layer (extension beyond the reference; include/kb_b200.h "Task layer") -------------------------
int kb_set_task(KbHandle* hh, const KbTaskDef* task, const double* target) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !task) return fail(KB_ERR_INVALID, "kb_set_task: null");
  if (task->mode != KB_TASK_CONST && task->mode != KB_TASK_OBJECT_TO_TARGET && task->mode != KB_TASK_SWARM_TO_TARGET)
    return fail(KB_ERR_INVALID, "kb_set_task: unknown mode");
  const int minM = *std::min_element(h->hostNumObjects.begin(), h->hostNumObjects.end());
  const int minN = *std::min_element(h->hostNumKilobots.begin(), h->hostNumKilobots.end());
  if (task->mode == KB_TASK_OBJECT_TO_TARGET && (task->object < 0 || task->object >= minM))
    return fail(KB_ERR_INVALID, "kb_set_task: object index out of range (every scene of the batch must have the object)");
  if (task->mode == KB_TASK_SWARM_TO_TARGET && minN < 1) return fail(KB_ERR_INVALID, "kb_set_task: a scene without kilobots");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  const size_t E = (size_t)h->numEnvs;
  std::vector<double> ts(E * KB_TASK_WORDS, 0.0);
  if (!target) {  // keep the current targets
    CUDA_TRY(cudaMemcpy(ts.data(), h->dTask, sizeof(double) * ts.size(), cudaMemcpyDeviceToHost));
    for (size_t e = 0; e < E; ++e)
      for (int k = 3; k < KB_TASK_WORDS; ++k) ts[e * KB_TASK_WORDS + k] = 0.0;
  } else {
    for (size_t e = 0; e < E; ++e)
      for (int k = 0; k < 3; ++k) ts[e * KB_TASK_WORDS + k] = target[e * 3 + k];
  }
  CUDA_TRY(cudaMemcpy(h->dTask, ts.data(), sizeof(double) * ts.size(), cudaMemcpyHostToDevice));
  TaskConst& t = h->task;
  t.mode = task->mode;
  t.object = task->object;
  t.maxSteps = task->max_episode_steps;
  t.pad = 0;
  t.wPos = task->w_position;
  t.wAng = task->w_orientation;
  t.stepPenalty = task->step_penalty;
  t.bonus = task->success_bonus;
  t.posTol = task->position_tolerance;
  t.angTol = task->orientation_tolerance;
  return KB_OK;
}

int kb_get_episode_stats(KbHandle* hh, double* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !out) return fail(KB_ERR_INVALID, "kb_get_episode_stats: null");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  const size_t E = (size_t)h->numEnvs;
  std::vector<double> ts(E * KB_TASK_WORDS);
  CUDA_TRY(cudaMemcpy(ts.data(), h->dTask, sizeof(double) * ts.size(), cudaMemcpyDeviceToHost));
  for (size_t e = 0; e < E; ++e)
    for (int k = 0; k < KB_EPISODE_STATS; ++k) out[e * KB_EPISODE_STATS + k] = ts[e * KB_TASK_WORDS + 3 + k];
  return KB_OK;
}

int kb_reduce_episode_stats(KbHandle* hh, double* out_device, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !out_device) return fail(KB_ERR_INVALID, "kb_reduce_episode_stats: null");
  CUDA_TRY(cudaSetDevice(h->device));
  kb_reduce_stats_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(h->dTask, h->dBlobs, h->L.blobWords, h->L.oHdr + H_STATUS,
                                                              h->numEnvs, out_device);
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

int kb_bind_flat_observation(KbHandle* hh, float* obs_flat) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return fail(KB_ERR_INVALID, "kb_bind_flat_observation: null handle");
  h->obsFlat = obs_flat;
  return KB_OK;
}

int kb_flat_observation_dim(const KbHandle* hh) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  if (!h) return fail(KB_ERR_INVALID, "kb_flat_observation_dim: null handle");
  return 2 * h->L.N + h->L.L + 4 * h->L.M;
}

// ---- arithmetic self-test (kb_sqrt / kb_rcp / kb_div against the plain operators) -----------------------------
}  // extern "C"
namespace kb {
__device__ __forceinline__ uint32_t mixBits(uint32_t x) {   // (murmur3 finaliser: a bijection of the 32-bit words)
  x ^= x >> 16; x *= 0x85ebca6bu; x ^= x >> 13; x *= 0xc2b2ae35u; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ bool sameFloat(float a, float b) {
  return __float_as_uint(a) == __float_as_uint(b) || (a != a && b != b);
}
__global__ void kb_selftest_math_kernel(int divRounds, unsigned long long* mismatches) {
  unsigned long long bad0 = 0ull, bad1 = 0ull, bad2 = 0ull, taken = 0ull;
  const unsigned long long total = 1ull << 32;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const uint32_t u = (uint32_t)i;
    const float x = __uint_as_float(u);
    {
      bool out = false;
      const float y = kb_sqrt_u(x, out);
      if (!out && !sameFloat(y, sqrtf(x))) ++bad0;
      if (!out) ++taken;
      out = false;
      const float z = kb_rcp_u(x, out);
      if (!out && !sameFloat(z, 1.0f / x)) ++bad1;
      if (!out) ++taken;
    }
    for (int r = 0; r < divRounds; ++r) {
      uint32_t ua = mixBits(u ^ (0x9e3779b9u * (uint32_t)(2 * r + 1))), ub = mixBits(~u + 0x7f4a7c15u * (uint32_t)(r + 1));
      if ((r & 1) != 0) {   // both exponents inside the fast path's window
        ua = (ua & 0x807fffffu) | ((64u + ((ua >> 23) & 0xFFu) % 127u) << 23);
        ub = (ub & 0x807fffffu) | ((64u + ((ub >> 23) & 0xFFu) % 127u) << 23);
      }
      const float a = __uint_as_float(ua), b = __uint_as_float(ub);
      bool out = false;
      const float q = kb_div_u(a, b, out);
      if (!out && !sameFloat(q, a / b)) ++bad2;
      if (!out) ++taken;
    }
  }
  if (bad0) atomicAdd(mismatches + 0, bad0);
  if (bad1) atomicAdd(mismatches + 1, bad1);
  if (bad2) atomicAdd(mismatches + 2, bad2);
  atomicAdd(mismatches + 3, taken);
}
// The position solver's kilobot-kilobot step the way the kernels run it -- straight-line pass, rows stored, out-of-line exact
// pass if a range test fired -- against the plain-operator template on 2^26 pseudo-random pairs of bodies: ordinary
// overlaps and separations, coincident and nearly coincident centres (zero / denormal squared distances), huge
// coordinates (infinite squared distance), separations within a few ulps of the slop (tiny corrections), zero and huge
// inverse masses.  mismatches[4] counts differing rows or verdicts, mismatches[5] the cases that took the exact pass.
__global__ void kb_selftest_pair_kernel(unsigned long long* mismatches) {
  __shared__ float4 rows[2 * 256];
  unsigned long long bad = 0ull, cold = 0ull;
  const uint32_t wA = (uint32_t)__cvta_generic_to_shared(&rows[2 * threadIdx.x]), wB = wA + 16u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < (1u << 26); i += gridDim.x * blockDim.x) {
    const uint32_t h0 = mixBits(i * 2u + 1u), h1 = mixBits(h0 ^ 0x68bc21ebu), h2 = mixBits(h1 + 0x02e5be93u), h3 = mixBits(h2 ^ i);
    const float ux = (float)(h0 & 0xFFFFu) * (1.0f / 65536.0f), uy = (float)(h0 >> 16) * (1.0f / 65536.0f);
    const float ang = 6.2831853f * (float)(h1 & 0xFFFFu) * (1.0f / 65536.0f);
    const int kind = (int)(h1 >> 16) & 15;
    float dist = 0.5f + 0.4f * (float)(h2 & 0xFFFFu) * (1.0f / 65536.0f);     // radii 0.4125 each: |.| around the contact
    float scale = 1.0f;
    if (kind == 0) dist = 0.0f;
    else if (kind == 1) dist = 1.0e-30f * ux;
    else if (kind == 2) dist = 1.0e-18f * (1.0f + uy);
    else if (kind == 3) scale = 3.0e19f;
    else if (kind == 4) dist = 0.825f - 0.005f + ((float)((int)(h2 >> 16) & 63) - 32.0f) * 5.9604645e-8f;
    float4 a0 = make_float4((ux * 40.0f - 20.0f) * scale, (uy * 30.0f - 15.0f) * scale, 0.3f * ux, 0.25f);
    float4 b0 = make_float4(a0.x + dist * cosf(ang), a0.y + dist * sinf(ang), -0.2f * uy, 0.5f);
    float mA = 33.0f + ux, iA = 380.0f + uy, mB = 33.0f + uy, iB = 380.0f + ux;
    if (kind == 5) { mA = 0.0f; iA = 0.0f; mB = 0.0f; iB = 0.0f; }
    if (kind == 6) { mA = 1.0e25f; mB = 1.0e25f; }
    const bool skipZero = (h3 & 1u) != 0u;
    const float baum = (h3 & 2u) != 0u ? KB_BAUMGARTE : KB_TOI_BAUMGARTE, limit = (h3 & 2u) != 0u ? -3.0f * KB_LINEAR_SLOP : -1.5f * KB_LINEAR_SLOP;
    // reference: the plain operators
    float4 ra, rb;
    bool rmoved, rbad = false;
    const bool rok = kb_position_pair_t<true>(a0, b0, 0.4125f, 0.4125f, mA, iA, mB, iB, baum, limit, skipZero, ra, rb, rmoved, rbad);
    if (!rmoved) { ra = a0; rb = b0; }
    // the kernels' sequence
    sts_f4(wA, a0);
    sts_f4(wB, b0);
    float4 a1, b1;
    bool moved, fbad = false;
    bool ok = kb_position_pair_t<false>(a0, b0, 0.4125f, 0.4125f, mA, iA, mB, iB, baum, limit, skipZero, a1, b1, moved, fbad);
    if (moved) {
      sts_f4(wA, a1);
      sts_f4(wB, b1);
    }
    if (fbad) {
      ok = kb_position_pair_cold(wA, wB, a0, b0, 0.4125f, 0.4125f, mA, iA, mB, iB, baum, limit, skipZero);
      ++cold;
    }
    const float4 ga = lds_f4(wA), gb = lds_f4(wB);
    const bool same = sameFloat(ga.x, ra.x) && sameFloat(ga.y, ra.y) && sameFloat(ga.z, ra.z) && sameFloat(ga.w, ra.w) &&
                      sameFloat(gb.x, rb.x) && sameFloat(gb.y, rb.y) && sameFloat(gb.z, rb.z) && sameFloat(gb.w, rb.w) && ok == rok;
    if (!same) ++bad;
  }
  if (bad) atomicAdd(mismatches + 4, bad);
  if (cold) atomicAdd(mismatches + 5, cold);
}
}  // namespace kb
extern "C" {
int kb_selftest_exact_math(int32_t device, int32_t div_rounds_log2, uint64_t* mismatches) {
  using namespace kb;
  if (!mismatches || div_rounds_log2 < 0 || div_rounds_log2 > 6) return fail(KB_ERR_INVALID, "kb_selftest_exact_math: invalid arguments");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count < 1) {
    cudaGetLastError();
    return fail(KB_ERR_NO_DEVICE, "kb_selftest_exact_math: no CUDA device");
  }
  if (device >= 0) CUDA_TRY(cudaSetDevice(device));
  unsigned long long* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, 6 * sizeof(unsigned long long)));
  CUDA_TRY(cudaMemset(d, 0, 6 * sizeof(unsigned long long)));
  kb_selftest_math_kernel<<<148 * 8, 256>>>(1 << div_rounds_log2, d);
  CUDA_TRY(cudaGetLastError());
  kb_selftest_pair_kernel<<<148 * 4, 256>>>(d);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(mismatches, d, 6 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaFree(d));
  return KB_OK;
}

// ---- geometry probe (kb_narrow.cuh, kb_toi.cuh one case at a time; the kernel is in kb_probe.cu) -------------------
}  // extern "C"
cudaError_t kbLaunchProbeGeometry(int op, int n, const void* px, const KbProbeCase* cases, uint32_t* out);
extern "C" {
int kb_probe_geometry(int32_t device, int32_t op, int32_t n, const KbProbeShape* shapes, int32_t num_shapes,
                      const KbProbeCase* cases, uint32_t* out) {
  using namespace kb;
  if (!shapes || num_shapes < 1 || !out || op < KB_PROBE_SHAPE || op > KB_PROBE_TOI || (op != KB_PROBE_SHAPE && (!cases || n < 0)))
    return fail(KB_ERR_INVALID, "kb_probe_geometry: invalid arguments");
  std::vector<ProxyConst> px((size_t)num_shapes);
  std::memset(px.data(), 0, sizeof(ProxyConst) * px.size());
  for (int s = 0; s < num_shapes; ++s) {
    const KbProbeShape& ps = shapes[s];
    if (ps.kind == KB_PROBE_EDGE) {
      if ((ps.wall_edges != 3 && ps.wall_edges != 4) || ps.edge < 0 || ps.edge >= ps.wall_edges)
        return fail(KB_ERR_INVALID, "kb_probe_geometry: bad chain edge");
      KbSceneDesc sd;
      std::memset(&sd, 0, sizeof(sd));
      sd.wall_x0 = ps.wall_x0; sd.wall_y0 = ps.wall_y0; sd.wall_x1 = ps.wall_x1; sd.wall_y1 = ps.wall_y1;
      sd.wall_edges = ps.wall_edges;
      buildChainEdge(sd, ps.edge, &px[s]);
    } else {
      const int rc = buildFixtureShape(ps.fixture, &px[s]);
      if (rc != KB_OK) return rc;
    }
  }
  if (op == KB_PROBE_SHAPE) {
    for (int s = 0; s < num_shapes; ++s) {
      const ProxyConst& pc = px[s];
      uint32_t* o = out + (size_t)s * KB_PROBE_OUT_WORDS;
      std::memset(o, 0, KB_PROBE_OUT_WORDS * 4);
      const float head[6] = {0.0f, pc.radius, 0.0f, 0.0f, pc.cx, pc.cy};
      std::memcpy(o, head, sizeof(head));
      o[0] = (uint32_t)(pc.type == SHAPE_EDGE ? 2 : (pc.type == SHAPE_CIRCLE ? 1 : pc.count));
      o[2] = (uint32_t)pc.has0;
      o[3] = (uint32_t)pc.has3;
      std::memcpy(o + 6, pc.vx, 4 * KB_MAX_POLY_VERTS);
      std::memcpy(o + 14, pc.vy, 4 * KB_MAX_POLY_VERTS);
      std::memcpy(o + 22, pc.nx, 4 * KB_MAX_POLY_VERTS);
      std::memcpy(o + 30, pc.ny, 4 * KB_MAX_POLY_VERTS);
    }
    return KB_OK;
  }
  for (int i = 0; i < n; ++i) {
    if (cases[i].a < 0 || cases[i].a >= num_shapes || cases[i].b < 0 || cases[i].b >= num_shapes)
      return fail(KB_ERR_INVALID, "kb_probe_geometry: shape index out of range");
    // the pairs the contact register forms (Sim::evaluate): A a circle only against a circle, B never an edge
    const int tA = px[cases[i].a].type, tB = px[cases[i].b].type;
    if (op == KB_PROBE_COLLIDE && (tB == SHAPE_EDGE || (tA == SHAPE_CIRCLE && tB != SHAPE_CIRCLE)))
      return fail(KB_ERR_INVALID, "kb_probe_geometry: no narrowphase routine for this pair of shapes");
  }
  if (n == 0) return KB_OK;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count < 1) {
    cudaGetLastError();
    return fail(KB_ERR_NO_DEVICE, "kb_probe_geometry: no CUDA device");
  }
  if (device >= 0) CUDA_TRY(cudaSetDevice(device));
  ProxyConst* dPx = nullptr;
  KbProbeCase* dCases = nullptr;
  uint32_t* dOut = nullptr;
  const size_t outBytes = (size_t)n * KB_PROBE_OUT_WORDS * 4;
  cudaError_t e = cudaMalloc(&dPx, sizeof(ProxyConst) * px.size());
  if (e == cudaSuccess) e = cudaMalloc(&dCases, sizeof(KbProbeCase) * (size_t)n);
  if (e == cudaSuccess) e = cudaMalloc(&dOut, outBytes);
  if (e == cudaSuccess) e = cudaMemcpy(dPx, px.data(), sizeof(ProxyConst) * px.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dCases, cases, sizeof(KbProbeCase) * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(dOut, 0, outBytes);
  if (e == cudaSuccess) {
    e = kbLaunchProbeGeometry(op, n, dPx, dCases, dOut);
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out, dOut, outBytes, cudaMemcpyDeviceToHost);
  cudaFree(dPx);
  cudaFree(dCases);
  cudaFree(dOut);
  if (e != cudaSuccess) return fail(KB_ERR_CUDA, std::string("kb_probe_geometry: ") + cudaGetErrorString(e));
  return KB_OK;
}

// ---- off-screen rasteriser (kb_render.cuh) ---------------------------------------------------------------
int kb_render(KbHandle* hh, const int32_t* env_ids, int32_t num_images, int32_t width, int32_t height, uint8_t* rgb,
              void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !env_ids || !rgb || num_images < 1 || width < 1 || height < 1)
    return fail(KB_ERR_INVALID, "kb_render: invalid arguments");
  if (num_images > 65535) return fail(KB_ERR_INVALID, "kb_render: at most 65535 images per call");
  for (int i = 0; i < num_images; ++i)
    if (env_ids[i] < 0 || env_ids[i] >= h->numEnvs) return fail(KB_ERR_INVALID, "kb_render: env id out of range");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (num_images > h->renderIdsCap) {
    CUDA_TRY(cudaStreamSynchronize(st));
    cudaFree(h->dRenderIds);
    h->dRenderIds = nullptr;
    CUDA_TRY(cudaMalloc(&h->dRenderIds, sizeof(int32_t) * (size_t)num_images));
    h->renderIdsCap = num_images;
  }
  CUDA_TRY(cudaMemcpyAsync(h->dRenderIds, env_ids, sizeof(int32_t) * (size_t)num_images, cudaMemcpyHostToDevice, st));
  RenderArgs a;
  a.L = h->L;
  a.blobs = h->dBlobs;
  a.envScene = h->dEnvScene;
  a.proxies = h->dProxies;
  a.bodies = h->dBodies;
  a.scenes = h->dScenes;
  a.lights = h->dLights;
  a.envIds = h->dRenderIds;
  a.numImages = num_images;
  a.width = width;
  a.height = height;
  a.x0 = h->wall[0]; a.y0 = h->wall[1]; a.x1 = h->wall[2]; a.y1 = h->wall[3];
  a.out = rgb;
  const dim3 block(16, 16), grid((width + 15) / 16, (height + 15) / 16, num_images);
  kb_render_kernel<<<grid, block, 0, st>>>(a);
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

// ---- per-kilobot local observations (kb_local.cuh) -----------------------------------------------------------------
static int localObsDim(const Handle* h, const KbLocalObsDef* def, const char* who) {
  if (!h) return fail(KB_ERR_INVALID, std::string(who) + ": null handle");
  if (!def) return fail(KB_ERR_INVALID, std::string(who) + ": null def");
  const int all = KB_LOCAL_NEIGHBOURS | KB_LOCAL_OBJECTS | KB_LOCAL_LIGHT;
  if (def->parts == 0 || (def->parts & ~all) != 0)
    return fail(KB_ERR_INVALID, std::string(who) + ": parts must be a non-empty set of KB_LOCAL_* bits");
  if (def->max_neighbours < 1 || def->max_neighbours > 32)
    return fail(KB_ERR_INVALID, std::string(who) + ": max_neighbours must be in 1..32");
  if (!std::isfinite(def->radius) || !(def->radius > 0.0f))
    return fail(KB_ERR_INVALID, std::string(who) + ": radius must be finite and > 0");
  if ((def->parts & KB_LOCAL_OBJECTS) && h->L.M == 0)
    return fail(KB_ERR_INVALID, std::string(who) + ": KB_LOCAL_OBJECTS on a batch without objects");
  if ((def->parts & KB_LOCAL_LIGHT) && h->L.numLights == 0)
    return fail(KB_ERR_INVALID, std::string(who) + ": KB_LOCAL_LIGHT on a batch without lights");
  int D = 0;
  if (def->parts & KB_LOCAL_NEIGHBOURS) D += 1 + 4 * def->max_neighbours;
  if (def->parts & KB_LOCAL_OBJECTS) D += 5 * h->L.M;
  if (def->parts & KB_LOCAL_LIGHT) D += 3;
  return D;
}

int kb_local_observation_dim(const KbHandle* hh, const KbLocalObsDef* def) {
  return localObsDim(reinterpret_cast<const Handle*>(hh), def, "kb_local_observation_dim");
}

int kb_local_observation(KbHandle* hh, const KbLocalObsDef* def, const uint8_t* mask, float* out, void* stream) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int D = localObsDim(h, def, "kb_local_observation");
  if (D < 0) return D;
  if (!out) return fail(KB_ERR_INVALID, "kb_local_observation: null out");
  if (h->numEnvs == 0 || h->L.N == 0) return KB_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  LocalArgs a;
  a.L = h->L;
  a.blobs = h->dBlobs;
  a.envScene = h->dEnvScene;
  a.bodies = h->dBodies;
  a.scenes = h->dScenes;
  a.lights = h->dLights;
  a.mask = mask;
  a.out = out;
  a.numEnvs = h->numEnvs;
  a.K = def->max_neighbours;
  a.parts = def->parts;
  a.D = D;
  a.r2 = def->radius * def->radius;
  // grid over the table (metres), cells at least 1.001 radius wide: the slack keeps a pair within the radius in adjacent
  // cells whatever the rounding of the cell index; a radius wider than the table leaves one cell (brute force)
  const double x0 = h->wall[0] / 25.0, y0 = h->wall[1] / 25.0;
  const double w = std::max(h->wall[2] / 25.0 - x0, h->wall[3] / 25.0 - y0);
  const double cw0 = 1.001 * (double)def->radius;
  int n = w > 0.0 ? (int)std::min((double)KB_LOCAL_GRID_AXIS, std::floor(w / cw0)) : 1;
  n = std::max(n, 1);
  const double cw = w > 0.0 ? w / n : 1.0;
  a.x0 = (float)x0;
  a.y0 = (float)y0;
  a.invCell = (float)(1.0 / cw);
  a.gx = n;
  a.gy = n;
  const bool forceGrid = [] {
    const char* ev = getenv("KB_LOCAL_FORCE_GRID");
    return ev && atoi(ev) != 0;
  }();
  cudaStream_t st = (cudaStream_t)stream;
  const bool small = a.K <= 8;
  if (!forceGrid && h->L.B <= KB_LOCAL_WARP_BODIES) {
    const int grid = (h->numEnvs + KB_LOCAL_WARPS - 1) / KB_LOCAL_WARPS;
    if (small)
      kb_local_warp_kernel<8><<<grid, 32 * KB_LOCAL_WARPS, 0, st>>>(a);
    else
      kb_local_warp_kernel<32><<<grid, 32 * KB_LOCAL_WARPS, 0, st>>>(a);
  } else {
    const int cells = a.gx * a.gy;
    const size_t smem = 16 * (size_t)h->L.B + 4 * (size_t)(2 * cells + 1) + 2 * (size_t)h->L.N;
    if (smem > 48 * 1024) CUDA_TRY(small ? raiseSmemLimit(kb_local_grid_kernel<8>, smem) : raiseSmemLimit(kb_local_grid_kernel<32>, smem));
    if (small)
      kb_local_grid_kernel<8><<<h->numEnvs, KB_LOCAL_CTA, smem, st>>>(a);
    else
      kb_local_grid_kernel<32><<<h->numEnvs, KB_LOCAL_CTA, smem, st>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  return KB_OK;
}

int kb_get_mass_data(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !out) return fail(KB_ERR_INVALID, "kb_get_mass_data: null");
  for (int s = 0; s < h->numScenes; ++s)
    for (int b = 0; b < h->L.B; ++b) {
      const BodyConst& bc = h->hostBodies[s][b];
      float* o = out + ((size_t)s * h->L.B + b) * 4;
      o[0] = bc.invMass; o[1] = bc.invI; o[2] = bc.lcx; o[3] = bc.lcy;
    }
  return KB_OK;
}

}  // extern "C"
