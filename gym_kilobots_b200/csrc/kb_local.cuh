// Per-kilobot local observations (include/kb_b200.h kb_local_observation): for every present kilobot of an env, its
// neighbours within a radius, the env's objects and the light at its sensor, all in the kilobot's own frame.  Read-only
// consumer of the per-env state blobs of either tier (transforms, light state, header word H_SCENE), the per-scene body
// kinds and light constants; it never touches the physics.  Two launch shapes with one result:
//   - kb_local_warp_kernel: a warp per env, brute-force scan over the env's kilobots staged in shared memory (batches of
//     up to KB_LOCAL_WARP_BODIES bodies: C2, C3, C5, the lane-group tier);
//   - kb_local_grid_kernel: a CTA per env, a uniform grid (cell >= radius) built by a counting sort with warp-aggregated
//     shared atomics, and a 3 x 3 cell scan per kilobot (large swarms; every batch with KB_LOCAL_FORCE_GRID=1).
// Neighbours are kept in a sorted register list of 64-bit keys (d2 bits << 32 | padded index): d2 >= 0, so the key order
// is the (d2, j) order of the contract and the result does not depend on the order in which candidates are visited.
// All float32 arithmetic is plain IEEE mul/add (the translation unit builds with -fmad=false), so
// gym_kilobots_b200/local_obs.py reproduces it bit for bit in numpy.
#pragma once
#include "kb_types.cuh"

namespace kb {

#define KB_LOCAL_WARP_BODIES 64   /* Bmax of the warp-per-env kernel (its per-warp staging area) */
#define KB_LOCAL_GRID_AXIS 32     /* most grid cells per axis */
#define KB_LOCAL_CTA 256          /* threads of the grid kernel's CTA */
#define KB_LOCAL_WARPS 4          /* envs (warps) per block of the warp kernel */

struct LocalArgs {
  Layout L;
  const float* blobs;
  const int32_t* envScene;     // null: every env is on scene 0
  const BodyConst* bodies;     // [scene][L.Bp]
  const SceneConst* scenes;
  const LightConst* lights;    // [scene][max(L.numLights, 1)]
  const uint8_t* mask;         // [E] or null
  float* out;                  // [E][L.N][D]
  int32_t numEnvs, K, parts, D;
  float r2;
  // grid of kb_local_grid_kernel, metres: cell (x, y) covers [x0 + x / invCell, ...), indices clamped to the grid
  int32_t gx, gy;
  float x0, y0, invCell;
};

__device__ __forceinline__ float obsCoord(float b2) { return (float)((double)b2 / 25.0); }

// the K smallest keys seen so far, ascending (unused slots hold ~0)
template <int KC>
struct TopK {
  unsigned long long k[KC];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int i = 0; i < KC; ++i) k[i] = ~0ull;
  }
  __device__ __forceinline__ void push(unsigned long long c) {
    if (c >= k[KC - 1]) return;
#pragma unroll
    for (int i = KC - 1; i > 0; --i) k[i] = c < k[i - 1] ? k[i - 1] : (c < k[i] ? c : k[i]);
    k[0] = c < k[0] ? c : k[0];
  }
};

// neighbour candidate j of kilobot i (both present, j != i)
template <int KC>
__device__ __forceinline__ void visit(const float4 pi, const float4 pj, int j, float r2, int& count, TopK<KC>& t) {
  const float dx = pj.x - pi.x, dy = pj.y - pi.y;
  const float d2 = dx * dx + dy * dy;
  if (d2 <= r2) {
    ++count;
    t.push(((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)j);
  }
}

// lightValueGrad of kb_env.cuh on global memory: value and gradient of one light at (sx, sy), metres
__device__ __forceinline__ void localLightValueGrad(const LightConst& lc, const double* ls, double sx, double sy, double* value,
                                                    double* gx, double* gy) {
  if (lc.type == KB_LIGHT_LINEAR) {
    const double2 sc = kb_sincosd(ls[0]);
    *value = sc.y * sx + sc.x * sy;
    *gx = sc.y;
    *gy = sc.x;
    return;
  }
  double g0 = -1 * (sx - ls[0]);
  double g1 = -1 * (sy - ls[1]);
  const double norm = sqrt(g0 * g0 + g1 * g1);
  double v = 1.0;
  v -= norm / lc.radius;
  v = v < 1. ? v : 1.;
  v = v > .0 ? v : .0;
  v *= 255;
  if (norm == 0.0) {
    g0 = 0.0;
    g1 = 0.0;
  } else {
    g0 /= norm;
    g1 /= norm;
  }
  if (norm > lc.radius) {
    g0 *= .0;
    g1 *= .0;
  }
  *value = v;
  *gx = g0;
  *gy = g1;
}

// one kilobot's row.  xs: the env's staged bodies (x m, y m, sin, cos), objects at 0..L.M-1, kilobot k at L.M + k.
template <int KC>
__device__ __forceinline__ void emitRow(const LocalArgs& a, const float* blob, int scene, int numObjects, int i,
                                        const float4* xs, int count, const TopK<KC>& t, float* row) {
  const Layout& L = a.L;
  const float4 pi = xs[L.M + i];
  int col = 0;
  if (a.parts & KB_LOCAL_NEIGHBOURS) {
    row[col++] = (float)count;
#pragma unroll
    for (int s = 0; s < KC; ++s) {
      if (s < a.K) {
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (t.k[s] != ~0ull) {
          const float4 pj = xs[L.M + (int)(uint32_t)t.k[s]];
          const float dx = pj.x - pi.x, dy = pj.y - pi.y;
          v = make_float4(pi.w * dx + pi.z * dy, -pi.z * dx + pi.w * dy, sqrtf(__uint_as_float((uint32_t)(t.k[s] >> 32))), 1.0f);
        }
        row[col] = v.x;
        row[col + 1] = v.y;
        row[col + 2] = v.z;
        row[col + 3] = v.w;
        col += 4;
      }
    }
  }
  if (a.parts & KB_LOCAL_OBJECTS) {
#pragma unroll 1
    for (int j = 0; j < L.M; ++j, col += 5) {
      if (j < numObjects) {
        const float4 pj = xs[j];
        const float dx = pj.x - pi.x, dy = pj.y - pi.y;
        row[col] = pi.w * dx + pi.z * dy;
        row[col + 1] = -pi.z * dx + pi.w * dy;
        row[col + 2] = pj.w * pi.w + pj.z * pi.z;
        row[col + 3] = pj.z * pi.w - pj.w * pi.z;
        row[col + 4] = 1.0f;
      } else {
        for (int c = 0; c < 5; ++c) row[col + c] = 0.0f;
      }
    }
  }
  if (a.parts & KB_LOCAL_LIGHT) {
    // the sensor point of senseControl (kb_env.cuh): the body origin of a SimplePhototaxisKilobot, else the rear point
    const float4 x = reinterpret_cast<const float4*>(blob + L.oXf)[L.M + i];
    const int kind = __ldg(&a.bodies[(size_t)scene * L.Bp + L.M + i].kind);
    double sx, sy;
    if (kind == KB_KILOBOT_SIMPLE_PHOTOTAXIS) {
      sx = (double)x.x / 25.0;
      sy = (double)x.y / 25.0;
    } else {
      Xf xf;
      xf.p = mk(x.x, x.y);
      xf.q.s = x.z;
      xf.q.c = x.w;
      const V2 wp = xmul(xf, mk((float)(25.0 * 0.0), (float)(25.0 * -0.0165)));
      sx = (double)wp.x / 25.0;
      sy = (double)wp.y / 25.0;
    }
    const LightConst* lc = a.lights + (size_t)scene * L.numLights;
    const double* ls = reinterpret_cast<const double*>(blob + L.oLight);
    double value = 0.0, gx = 0.0, gy = 0.0;
    if (L.numLights == 1) {
      localLightValueGrad(lc[0], ls, sx, sy, &value, &gx, &gy);
    } else {
      double best = 0.0;
      int so = 0;
      for (int l = 0; l < L.numLights; ++l) {
        double v, g0, g1;
        localLightValueGrad(lc[l], ls + so, sx, sy, &v, &g0, &g1);
        value += v;
        if (l == 0 || v > best) {
          best = v;
          gx = g0;
          gy = g1;
        }
        so += lc[l].type == KB_LIGHT_MOMENTUM ? 4 : (lc[l].type == KB_LIGHT_LINEAR ? 1 : 2);
      }
    }
    const double c = (double)x.w, s = (double)x.z;
    row[col] = (float)value;
    row[col + 1] = (float)(c * gx + s * gy);
    row[col + 2] = (float)(-s * gx + c * gy);
  }
}

__device__ __forceinline__ void nanRow(const LocalArgs& a, float* row) {
  for (int c = 0; c < a.D; ++c) row[c] = __int_as_float(0x7FC00000);
}

__device__ __forceinline__ float4 stageBody(const float* blob, const Layout& L, int b) {
  const float4 x = reinterpret_cast<const float4*>(blob + L.oXf)[b];
  return make_float4(obsCoord(x.x), obsCoord(x.y), x.z, x.w);
}

__device__ __forceinline__ int localScene(const LocalArgs& a, const float* blob) {
  return a.envScene ? (int)reinterpret_cast<const uint32_t*>(blob)[a.L.oHdr + H_SCENE] : 0;
}

// ---- a warp per env, brute force (L.B <= KB_LOCAL_WARP_BODIES)
template <int KC>
__global__ void __launch_bounds__(32 * KB_LOCAL_WARPS) kb_local_warp_kernel(const __grid_constant__ LocalArgs a) {
  __shared__ float4 stage[KB_LOCAL_WARPS][KB_LOCAL_WARP_BODIES];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int env = blockIdx.x * KB_LOCAL_WARPS + w;
  if (env >= a.numEnvs || (a.mask && !a.mask[env])) return;   // whole warps only: no block-wide barrier follows
  const Layout& L = a.L;
  const float* blob = a.blobs + (size_t)env * L.blobWords;
  const int scene = localScene(a, blob);
  const int numObjects = __ldg(&a.scenes[scene].numObjects), numKilobots = __ldg(&a.scenes[scene].numKilobots);
  float4* xs = stage[w];
  for (int b = lane; b < L.B; b += 32) xs[b] = stageBody(blob, L, b);
  __syncwarp();
#pragma unroll 1
  for (int i = lane; i < L.N; i += 32) {
    float* row = a.out + ((size_t)env * L.N + i) * a.D;
    if (i >= numKilobots) {
      nanRow(a, row);
      continue;
    }
    TopK<KC> t;
    t.init();
    int count = 0;
    if (a.parts & KB_LOCAL_NEIGHBOURS) {
      const float4 pi = xs[L.M + i];
#pragma unroll 1
      for (int j = 0; j < numKilobots; ++j)
        if (j != i) visit(pi, xs[L.M + j], j, a.r2, count, t);
    }
    emitRow(a, blob, scene, numObjects, i, xs, count, t, row);
  }
}

// grid cell of a position, clamped (a NaN lands in cell 0 and never passes d2 <= r2)
__device__ __forceinline__ int2 localCell(const LocalArgs& a, float4 p) {
  const float tx = fminf(fmaxf((p.x - a.x0) * a.invCell, 0.0f), (float)(a.gx - 1));
  const float ty = fminf(fmaxf((p.y - a.y0) * a.invCell, 0.0f), (float)(a.gy - 1));
  return make_int2((int)tx, (int)ty);
}

// ---- a CTA per env, uniform grid.  Dynamic shared memory: float4 xs[L.B], int start[cells + 1], int cur[cells],
// u16 sorted[L.N]
template <int KC>
__global__ void __launch_bounds__(KB_LOCAL_CTA) kb_local_grid_kernel(const __grid_constant__ LocalArgs a) {
  extern __shared__ float4 kb_local_smem[];
  const int env = blockIdx.x;
  if (a.mask && !a.mask[env]) return;   // the whole CTA
  const Layout& L = a.L;
  const int tid = threadIdx.x, lane = tid & 31;
  const int cells = a.gx * a.gy;
  float4* xs = kb_local_smem;
  int* start = reinterpret_cast<int*>(xs + L.B);
  int* cur = start + cells + 1;
  uint16_t* sorted = reinterpret_cast<uint16_t*>(cur + cells);
  __shared__ int warpSum[KB_LOCAL_CTA / 32];
  const float* blob = a.blobs + (size_t)env * L.blobWords;
  const int scene = localScene(a, blob);
  const int numObjects = __ldg(&a.scenes[scene].numObjects), numKilobots = __ldg(&a.scenes[scene].numKilobots);
  for (int b = tid; b < L.B; b += KB_LOCAL_CTA) xs[b] = stageBody(blob, L, b);
  for (int c = tid; c < cells; c += KB_LOCAL_CTA) cur[c] = 0;
  __syncthreads();
  const bool nb = (a.parts & KB_LOCAL_NEIGHBOURS) != 0;
  if (nb) {
    const unsigned lt = (1u << lane) - 1u;
    // counting sort of the present kilobots by cell; a warp's lanes of one cell share one shared atomic
    for (int base = 0; base < numKilobots; base += KB_LOCAL_CTA) {
      const int i = base + tid;
      int c = -1;
      if (i < numKilobots) {
        const int2 q = localCell(a, xs[L.M + i]);
        c = q.y * a.gx + q.x;
      }
      const unsigned m = __match_any_sync(0xFFFFFFFFu, c);
      if (c >= 0 && (m & lt) == 0u) atomicAdd(&cur[c], __popc(m));
    }
    __syncthreads();
    // exclusive scan of the counts: each thread takes a run of consecutive cells
    const int per = (cells + KB_LOCAL_CTA - 1) / KB_LOCAL_CTA;
    const int c0 = min(tid * per, cells), c1 = min(c0 + per, cells);
    int sum = 0;
    for (int c = c0; c < c1; ++c) sum += cur[c];
    int x = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xFFFFFFFFu, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warpSum[tid >> 5] = x;
    __syncthreads();
    int off = x - sum;
    for (int w = 0; w < (tid >> 5); ++w) off += warpSum[w];
    for (int c = c0; c < c1; ++c) {
      const int n = cur[c];
      start[c] = off;
      cur[c] = off;
      off += n;
    }
    if (tid == 0) start[cells] = numKilobots;
    __syncthreads();
    for (int base = 0; base < numKilobots; base += KB_LOCAL_CTA) {
      const int i = base + tid;
      int c = -1;
      if (i < numKilobots) {
        const int2 q = localCell(a, xs[L.M + i]);
        c = q.y * a.gx + q.x;
      }
      const unsigned m = __match_any_sync(0xFFFFFFFFu, c);
      const int leader = __ffs(m) - 1;
      int slot = 0;
      if (c >= 0 && lane == leader) slot = atomicAdd(&cur[c], __popc(m));
      slot = __shfl_sync(0xFFFFFFFFu, slot, leader);
      if (c >= 0) sorted[slot + __popc(m & lt)] = (uint16_t)i;
    }
    __syncthreads();
  }
#pragma unroll 1
  for (int i = tid; i < L.N; i += KB_LOCAL_CTA) {
    float* row = a.out + ((size_t)env * L.N + i) * a.D;
    if (i >= numKilobots) {
      nanRow(a, row);
      continue;
    }
    TopK<KC> t;
    t.init();
    int count = 0;
    if (nb) {
      const float4 pi = xs[L.M + i];
      const int2 q = localCell(a, pi);
#pragma unroll 1
      for (int cy = max(q.y - 1, 0); cy <= min(q.y + 1, a.gy - 1); ++cy) {
        const int cx0 = max(q.x - 1, 0), cx1 = min(q.x + 1, a.gx - 1);
        // the cells cx0..cx1 of one row are consecutive in the sorted list
#pragma unroll 1
        for (int p = start[cy * a.gx + cx0]; p < start[cy * a.gx + cx1 + 1]; ++p) {
          const int j = sorted[p];
          if (j != i) visit(pi, xs[L.M + j], j, a.r2, count, t);
        }
      }
    }
    emitRow(a, blob, scene, numObjects, i, xs, count, t, row);
  }
}

}  // namespace kb
