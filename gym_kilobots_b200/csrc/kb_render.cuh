// Off-screen rasteriser (SURVEY.md 8(f) n4): what KilobotsEnv.render draws through kb_rendering.KilobotsViewer
// (gym_kilobots/envs/kilobots_env.py:221-275; kb_rendering.py:7-113), evaluated per pixel straight from the
// per-env state blobs -- table, objects (lib/body.py:156-157,202-203,279-281), kilobots
// (lib/kilobot.py:129-145,205-210) and the light (lib/light.py:95-96,194-195).  No pygame surface, no host
// round trip: one thread per pixel, painter's order, uint8 RGB out.  Debug/video consumer of the state, not part
// of the step's timed path.  All arithmetic is float32 without FMA; oracle/kbo_env.cpp kbo_render mirrors it.
#pragma once
#include "kb_types.cuh"

namespace kb {

struct RenderArgs {
  Layout L;
  const float* blobs;
  const int32_t* envScene;
  const ProxyConst* proxies;
  const BodyConst* bodies;
  const SceneConst* scenes;
  const LightConst* lights;
  const int32_t* envIds;     // [numImages] device
  int32_t numImages, width, height;
  float x0, y0, x1, y1;      // world window in b2 units (metres * 25)
  uint8_t* out;              // [numImages][height][width][3]
};

struct Rgb {
  float r, g, b;
};

// one pixel; p in b2 units.  xf[b] = (p.x, p.y, sin, cos) of body b.
__device__ __forceinline__ Rgb shadePixel(const RenderArgs& a, const float4* xf, const double* light, const ProxyConst* px,
                                          const BodyConst* bc, const LightConst* lights, int numProxies, int wallEdges, float x, float y) {
  const float S = 25.0f;
  Rgb c = {255.0f, 255.0f, 255.0f};                                   // table, kilobots_env.py:254-255
  // border polyline, width .003 m (:256-257), never thinner than one pixel (pygame's minimum line width)
  const float hbx = fmaxf(0.0015f * S, (a.x1 - a.x0) / (float)a.width);
  const float hby = fmaxf(0.0015f * S, (a.y1 - a.y0) / (float)a.height);
  if (x - a.x0 < hbx || a.x1 - x < hbx || y - a.y0 < hby || a.y1 - y < hby) c = Rgb{0.0f, 0.0f, 0.0f};
  // objects, creation order (:261-262); proxies of the table come first
  for (int p = wallEdges; p < numProxies; ++p) {
    const int b = px[p].body;
    if (b >= a.L.M) break;
    const float4 t = xf[b];
    const float dx = x - t.x, dy = y - t.y;
    bool inside;
    if (px[p].type == SHAPE_CIRCLE) {
      inside = dx * dx + dy * dy <= px[p].radius * px[p].radius;
    } else {
      const float lx = t.w * dx + t.z * dy, ly = -t.z * dx + t.w * dy;  // b2MulT(q, d)
      inside = true;
      for (int i = 0; i < px[p].count; ++i)
        inside = inside && (px[p].nx[i] * (lx - px[p].vx[i]) + px[p].ny[i] * (ly - px[p].vy[i]) <= 0.0f);
    }
    if (inside) c = Rgb{93.0f, 133.0f, 195.0f};                       // lib/body.py:21
  }
  // kilobots (:265-266): disc r + .002, grey ring of width .005 drawn inwards, white heading line of width .005
  for (int b = a.L.M; b < a.L.B; ++b) {
    if (bc[b].kind == KB_BODY_ABSENT) continue;   // a padded index the env's scene does not populate
    const float4 t = xf[b];
    const float dx = x - t.x, dy = y - t.y;
    const float d2 = dx * dx + dy * dy;
    const float R = (0.0165f + 0.002f) * S, Rin = (0.0165f + 0.002f - 0.005f) * S;
    if (d2 > R * R) continue;
    c = Rgb{150.0f, 150.0f, 150.0f};
    if (d2 >= Rin * Rin) c = Rgb{100.0f, 100.0f, 100.0f};
    if (bc[b].kind != KB_KILOBOT_SIMPLE_PHOTOTAXIS) {
      const float lx = t.w * dx + t.z * dy, ly = -t.z * dx + t.w * dy;
      const float front = (0.0165f - 0.005f) * S, hw = 0.0025f * S;
      if (lx >= 0.0f && lx <= front && ly >= -hw && ly <= hw) c = Rgb{255.0f, 255.0f, 255.0f};
    }
  }
  // light (:269-270): CircularGradientLight / MomentumLight = translucent disc (255, 255, 30, alpha 150)
  int off = 0;
  for (int l = 0; l < a.L.numLights; ++l) {
    const int type = lights[l].type;
    if (type == KB_LIGHT_LINEAR) {
      off += 1;
      continue;
    }
    const float lx = (float)(light[off] * 25.0), ly = (float)(light[off + 1] * 25.0);
    const float R = (float)(lights[l].radius * 25.0);
    const float dx = x - lx, dy = y - ly;
    if (dx * dx + dy * dy <= R * R) {
      const float al = 150.0f / 255.0f, be = 1.0f - 150.0f / 255.0f;
      c = Rgb{255.0f * al + c.r * be, 255.0f * al + c.g * be, 30.0f * al + c.b * be};
    }
    off += type == KB_LIGHT_MOMENTUM ? 4 : 2;
  }
  return c;
}

__global__ void __launch_bounds__(256) kb_render_kernel(const RenderArgs a) {
  __shared__ float4 xf[KB_MAX_BODIES + 2];
  const int img = blockIdx.z;
  const int env = a.envIds[img];
  const float* blob = a.blobs + (size_t)env * a.L.blobWords;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  // transforms staged in shared memory for the lane-group tier (<= 62 bodies); a large swarm is read through L2
  const bool staged = a.L.B <= KB_MAX_BODIES;
  if (staged)
    for (int b = tid; b < a.L.B; b += blockDim.x * blockDim.y)
      xf[b] = *reinterpret_cast<const float4*>(blob + a.L.oXf + 4 * b);
  __syncthreads();
  const float4* xfp = staged ? xf : reinterpret_cast<const float4*>(blob + a.L.oXf);
  const int px_ = blockIdx.x * blockDim.x + threadIdx.x, py = blockIdx.y * blockDim.y + threadIdx.y;
  if (px_ >= a.width || py >= a.height) return;
  const int scene = a.envScene ? (int)reinterpret_cast<const uint32_t*>(blob)[a.L.oHdr + H_SCENE] : 0;   // (last reset's)
  const float x = a.x0 + ((float)px_ + 0.5f) * ((a.x1 - a.x0) / (float)a.width);
  const float y = a.y1 - ((float)py + 0.5f) * ((a.y1 - a.y0) / (float)a.height);   // image row 0 = top
  const Rgb c = shadePixel(a, xfp, reinterpret_cast<const double*>(blob + a.L.oLight), a.proxies + (size_t)scene * a.L.Pp,
                           a.bodies + (size_t)scene * a.L.Bp, a.lights + (size_t)scene * (a.L.numLights > 0 ? a.L.numLights : 1),
                           a.scenes[scene].numProxies, a.scenes[scene].wallEdges, x, y);
  uint8_t* o = a.out + (((size_t)img * a.height + py) * a.width + px_) * 3;
  o[0] = (uint8_t)(int)(c.r + 0.5f);
  o[1] = (uint8_t)(int)(c.g + 0.5f);
  o[2] = (uint8_t)(int)(c.b + 0.5f);
}

}  // namespace kb
