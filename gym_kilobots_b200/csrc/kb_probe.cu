// kb_probe.cu -- the kernel of kb_probe_geometry (include/kb_b200.h): the narrowphase, distance and time-of-impact
// device functions of kb_narrow.cuh / kb_toi.cuh, one case per thread, for the tests that compare them with float64
// geometry and with the oracle.  A translation unit of its own: ptxas compiles the out-of-line device functions
// (collide_polygons, time_of_impact, ...) for the call graph of their module, so a caller in kb_b200.cu would change the
// code of the step kernels.  The headers' out-of-line functions have host-side symbols too: inside an unnamed namespace
// this module's copies do not collide with kb_b200.cu's at link time.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kb_b200.h"

// Every header the kernel headers include must already be included above: its include guard then keeps it out of the
// unnamed namespace.  A new system header in kb_types.cuh (or below it) belongs in this list too.
namespace {
#include "kb_toi.cuh"
}  // namespace

namespace {
namespace kb {

__device__ __forceinline__ Xf probeXf(const float* x) {
  Xf xf;
  xf.p = mk(x[0], x[1]);
  xf.q.s = x[2];
  xf.q.c = x[3];
  return xf;
}
__device__ __forceinline__ SweepD probeSweep(const float* s, int fixedRot) {
  SweepD sw;
  sw.lc = mk(s[0], s[1]);
  sw.c0 = mk(s[2], s[3]);
  sw.c = mk(s[4], s[5]);
  sw.a0 = s[6];
  sw.a = s[7];
  sw.alpha0 = 0.0f;
  sw.fixedRot = fixedRot;
  return sw;
}
__global__ void kb_probe_geometry_kernel(int op, int n, const ProxyConst* __restrict__ px, const KbProbeCase* __restrict__ cases,
                                         uint32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const KbProbeCase& c = cases[i];
  const ProxyConst* A = px + c.a;
  const ProxyConst* Bp = px + c.b;
  const int tA = __ldg(&A->type), tB = __ldg(&Bp->type);
  uint32_t* o = out + (size_t)i * KB_PROBE_OUT_WORDS;
  if (op == KB_PROBE_COLLIDE) {
    // the dispatch of Sim::evaluate (kb_step.cuh)
    const Xf xfA = probeXf(c.xf_a), xfB = probeXf(c.xf_b);
    Manifold m;
    m.pointCount = 0;
    m.type = 0;
    m.lnx = m.lny = m.lpx = m.lpy = 0.0f;
    m.px[0] = m.py[0] = m.px[1] = m.py[1] = 0.0f;
    m.id[0] = m.id[1] = 0u;
    if (tB == SHAPE_CIRCLE) {
      if (tA == SHAPE_CIRCLE) collide_circles(m, __ldg(&A->radius), xfA, __ldg(&Bp->radius), xfB);
      else if (tA == SHAPE_POLYGON) collide_polygon_circle(m, A, xfA, __ldg(&Bp->radius), xfB);
      else collide_edge_circle(m, A, xfA, __ldg(&Bp->radius), xfB);
    } else {
      if (tA == SHAPE_POLYGON) collide_polygons(m, A, xfA, Bp, xfB);
      else collide_edge_polygon(m, A, xfA, Bp, xfB);
    }
    o[0] = (uint32_t)m.type;
    o[1] = (uint32_t)m.pointCount;
    o[2] = __float_as_uint(m.lnx); o[3] = __float_as_uint(m.lny);
    o[4] = __float_as_uint(m.lpx); o[5] = __float_as_uint(m.lpy);
    for (int k = 0; k < 2; ++k) {
      o[6 + 3 * k] = __float_as_uint(m.px[k]);
      o[7 + 3 * k] = __float_as_uint(m.py[k]);
      o[8 + 3 * k] = m.id[k];
    }
  } else if (op == KB_PROBE_DISTANCE) {
    DProxy pA, pB;
    pA.set(A);
    pB.set(Bp);
    SimplexCache cache;
    cache.metric = 0.0f;
    cache.count = 0;
    cache.iA0 = cache.iA1 = cache.iA2 = cache.iB0 = cache.iB1 = cache.iB2 = 0;
    const float d = gjk_distance(cache, pA, probeXf(c.xf_a), pB, probeXf(c.xf_b));
    o[0] = __float_as_uint(d);
    o[1] = (uint32_t)cache.count;
  } else if (op == KB_PROBE_TOI) {
    const SweepD sA = probeSweep(c.sweep_a, c.fixed_rot_a), sB = probeSweep(c.sweep_b, c.fixed_rot_b);
    o[0] = __float_as_uint(time_of_impact(A, sA, Bp, sB));
    o[1] = (tA == SHAPE_EDGE && tB == SHAPE_CIRCLE) ? __float_as_uint(time_of_impact_edge_circle(A, sA, Bp, sB)) : 0u;
    o[2] = __float_as_uint(time_of_impact(A, probeSweep(c.sweep_a, 0), Bp, probeSweep(c.sweep_b, 0)));
  }
}
}  // namespace kb
}  // namespace

// px: device kb::ProxyConst[] (kb_types.cuh)
cudaError_t kbLaunchProbeGeometry(int op, int n, const void* px, const KbProbeCase* cases, uint32_t* out) {
  kb::kb_probe_geometry_kernel<<<(n + 127) / 128, 128>>>(op, n, static_cast<const kb::ProxyConst*>(px), cases, out);
  return cudaGetLastError();
}
