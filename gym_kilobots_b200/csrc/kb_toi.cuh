// kb_toi.cuh -- continuous collision against the static table: GPU restatement of Box2D 2.3.x
// b2Distance (GJK + simplex cache), b2TimeOfImpact (conservative advancement) and
// b2World::SolveTOI / b2Island::SolveTOI (SURVEY.md Appendix B.8), reached from b2World.Step at
// gym_kilobots/envs/kilobots_env.py:187.  There are no bullets, so only dynamic-vs-table contacts
// are candidates.  One lane evaluates one candidate contact's time of impact; the (rare) TOI event
// itself -- a mini island of one dynamic body and its wall contacts -- is solved by lane 0.
#pragma once
#include "kb_step.cuh"

namespace kb {

struct SweepD {
  V2 lc, c0, c;
  float a0, a, alpha0;
  // the rotation of this sweep cannot influence the result, so b2Rot::Set (double-precision sin/cos here)
  // is skipped and q = (0, 1) is used: either a0 == a == 0, where (0, 1) IS the exact rotation (the table),
  // or the shape is a circle centred on a body whose local centre is zero (a kilobot), where q only ever
  // multiplies exact zeros and picks the support vertex of a one-vertex proxy
  int fixedRot;
};
__device__ __forceinline__ Xf sweep_xf(const SweepD& s, float beta) {
  Xf xf;
  xf.p = (1.0f - beta) * s.c0 + beta * s.c;
  float angle = (1.0f - beta) * s.a0 + beta * s.a;
  if (s.fixedRot) {
    xf.q.s = 0.0f;
    xf.q.c = 1.0f;
  } else {
    xf.q = rot_set(angle);
  }
  xf.p = xf.p - rmul(xf.q, s.lc);
  return xf;
}
__device__ __forceinline__ void sweep_normalize(SweepD& s) {
  float twoPi = 2.0f * KB_PI;
  float d = twoPi * floorf(s.a0 / twoPi);
  s.a0 -= d;
  s.a -= d;
}

// b2DistanceProxy over a scene proxy.  Three flavours with one interface: the generic one reads the template
// at run time; the edge and circle ones fix vertex count and vertex access at compile time, so that the by far
// most common continuous-collision pair (table edge against a kilobot) compiles to short straight-line code
// with its two edge vertices in registers -- same arithmetic, a fraction of the instructions and branches.
struct DProxy {
  const ProxyConst* pc;
  int type, count;
  float radius;
  __device__ __forceinline__ void set(const ProxyConst* p) {
    pc = p;
    type = __ldg(&p->type);
    radius = __ldg(&p->radius);
    count = type == SHAPE_CIRCLE ? 1 : (type == SHAPE_EDGE ? 2 : __ldg(&p->count));
  }
  __device__ __forceinline__ V2 vertex(int i) const {
    if (type == SHAPE_CIRCLE) return mk(0.0f, 0.0f);
    if (type == SHAPE_EDGE) return pvert(pc, 1 + i);
    return pvert(pc, i);
  }
  __device__ __forceinline__ int support(V2 d) const {
    int bestIndex = 0;
    float bestValue = dot(vertex(0), d);
    for (int i = 1; i < count; ++i) {
      float value = dot(vertex(i), d);
      if (value > bestValue) {
        bestIndex = i;
        bestValue = value;
      }
    }
    return bestIndex;
  }
};
struct DProxyEdge {
  V2 e1, e2;
  float radius;
  __device__ __forceinline__ void set(const ProxyConst* p) {
    e1 = pvert(p, 1);
    e2 = pvert(p, 2);
    radius = __ldg(&p->radius);
  }
  __device__ __forceinline__ V2 vertex(int i) const { return i == 0 ? e1 : e2; }
  __device__ __forceinline__ int support(V2 d) const {
    const float bestValue = dot(e1, d);
    const float value = dot(e2, d);
    return value > bestValue ? 1 : 0;
  }
};
struct DProxyCircle {
  float radius;
  __device__ __forceinline__ void set(const ProxyConst* p) { radius = __ldg(&p->radius); }
  __device__ __forceinline__ V2 vertex(int) const { return mk(0.0f, 0.0f); }
  __device__ __forceinline__ int support(V2 d) const {
    (void)dot(mk(0.0f, 0.0f), d);
    return 0;
  }
};

// Everything below is written without arrays, references into callers' frames or pointers to locals: the
// simplex, its cache and the separation function live in registers.  (Local memory is an L2 round trip in this
// kernel -- shared memory takes most of the L1 -- and b2Distance is a chain of dependent accesses.)
struct SimplexCache {
  float metric;
  int count;
  int iA0, iA1, iA2, iB0, iB1, iB2;
};
struct SimplexVertex {
  V2 wA, wB, w;
  float a;
  int indexA, indexB;
};

__device__ __forceinline__ float simplex_metric(int count, const SimplexVertex& v0, const SimplexVertex& v1,
                                                const SimplexVertex& v2) {
  if (count == 2) return length(v0.w - v1.w);
  if (count == 3) return cross(v1.w - v0.w, v2.w - v0.w);
  return 0.0f;
}
__device__ __forceinline__ void simplex_solve2(int& count, SimplexVertex& v0, SimplexVertex& v1) {
  V2 w1 = v0.w, w2 = v1.w;
  V2 e12 = w2 - w1;
  float d12_2 = -dot(w1, e12);
  if (d12_2 <= 0.0f) {
    v0.a = 1.0f;
    count = 1;
    return;
  }
  float d12_1 = dot(w2, e12);
  if (d12_1 <= 0.0f) {
    v1.a = 1.0f;
    count = 1;
    v0 = v1;
    return;
  }
  float inv_d12 = 1.0f / (d12_1 + d12_2);
  v0.a = d12_1 * inv_d12;
  v1.a = d12_2 * inv_d12;
  count = 2;
}
__device__ __forceinline__ void simplex_solve3(int& count, SimplexVertex& v0, SimplexVertex& v1, SimplexVertex& v2) {
  V2 w1 = v0.w, w2 = v1.w, w3 = v2.w;
  V2 e12 = w2 - w1;
  float w1e12 = dot(w1, e12);
  float w2e12 = dot(w2, e12);
  float d12_1 = w2e12;
  float d12_2 = -w1e12;
  V2 e13 = w3 - w1;
  float w1e13 = dot(w1, e13);
  float w3e13 = dot(w3, e13);
  float d13_1 = w3e13;
  float d13_2 = -w1e13;
  V2 e23 = w3 - w2;
  float w2e23 = dot(w2, e23);
  float w3e23 = dot(w3, e23);
  float d23_1 = w3e23;
  float d23_2 = -w2e23;
  float n123 = cross(e12, e13);
  float d123_1 = n123 * cross(w2, w3);
  float d123_2 = n123 * cross(w3, w1);
  float d123_3 = n123 * cross(w1, w2);
  if (d12_2 <= 0.0f && d13_2 <= 0.0f) {
    v0.a = 1.0f;
    count = 1;
    return;
  }
  if (d12_1 > 0.0f && d12_2 > 0.0f && d123_3 <= 0.0f) {
    float inv_d12 = 1.0f / (d12_1 + d12_2);
    v0.a = d12_1 * inv_d12;
    v1.a = d12_2 * inv_d12;
    count = 2;
    return;
  }
  if (d13_1 > 0.0f && d13_2 > 0.0f && d123_2 <= 0.0f) {
    float inv_d13 = 1.0f / (d13_1 + d13_2);
    v0.a = d13_1 * inv_d13;
    v2.a = d13_2 * inv_d13;
    count = 2;
    v1 = v2;
    return;
  }
  if (d12_1 <= 0.0f && d23_2 <= 0.0f) {
    v1.a = 1.0f;
    count = 1;
    v0 = v1;
    return;
  }
  if (d13_1 <= 0.0f && d23_1 <= 0.0f) {
    v2.a = 1.0f;
    count = 1;
    v0 = v2;
    return;
  }
  if (d23_1 > 0.0f && d23_2 > 0.0f && d123_1 <= 0.0f) {
    float inv_d23 = 1.0f / (d23_1 + d23_2);
    v1.a = d23_1 * inv_d23;
    v2.a = d23_2 * inv_d23;
    count = 2;
    v0 = v2;
    return;
  }
  float inv_d123 = 1.0f / (d123_1 + d123_2 + d123_3);
  v0.a = d123_1 * inv_d123;
  v1.a = d123_2 * inv_d123;
  v2.a = d123_3 * inv_d123;
  count = 3;
}

template <class PA, class PB>
__device__ __forceinline__ SimplexVertex simplex_vertex(const PA& pA, Xf tA, const PB& pB, Xf tB, int ia, int ib) {
  SimplexVertex sv;
  sv.indexA = ia;
  sv.indexB = ib;
  sv.wA = xmul(tA, pA.vertex(ia));
  sv.wB = xmul(tB, pB.vertex(ib));
  sv.w = sv.wB - sv.wA;
  sv.a = 0.0f;
  return sv;
}

// b2Distance(useRadii = false): distance between the core shapes; updates the cache.
template <class PA, class PB>
__device__ __forceinline__ float gjk_distance(SimplexCache& cache, const PA& pA, Xf tA, const PB& pB, Xf tB) {
  SimplexVertex v0, v1, v2;
  int count = cache.count;
  v0 = simplex_vertex(pA, tA, pB, tB, count > 0 ? cache.iA0 : 0, count > 0 ? cache.iB0 : 0);
  v1 = v0;
  v2 = v0;
  if (count > 1) v1 = simplex_vertex(pA, tA, pB, tB, cache.iA1, cache.iB1);
  if (count > 2) v2 = simplex_vertex(pA, tA, pB, tB, cache.iA2, cache.iB2);
  if (count > 1) {
    float metric1 = cache.metric;
    float metric2 = simplex_metric(count, v0, v1, v2);
    if (metric2 < 0.5f * metric1 || 2.0f * metric1 < metric2 || metric2 < KB_EPS) count = 0;
  }
  if (count == 0) {
    v0 = simplex_vertex(pA, tA, pB, tB, 0, 0);
    v0.a = 1.0f;
    count = 1;
  }
  const int k_maxIters = 20;
  int iter = 0;
  while (iter < k_maxIters) {
    const int saveCount = count;
    const int sA0 = v0.indexA, sB0 = v0.indexB, sA1 = v1.indexA, sB1 = v1.indexB, sA2 = v2.indexA, sB2 = v2.indexB;
    if (count == 2) simplex_solve2(count, v0, v1);
    else if (count == 3) simplex_solve3(count, v0, v1, v2);
    if (count == 3) break;
    // search direction
    V2 d;
    if (count == 1) {
      d = -v0.w;
    } else {
      V2 e12 = v1.w - v0.w;
      float sgn = cross(e12, -v0.w);
      d = sgn > 0.0f ? cross(1.0f, e12) : cross(e12, 1.0f);
    }
    if (dot(d, d) < KB_EPS * KB_EPS) break;
    SimplexVertex nv;
    nv.indexA = pA.support(rmulT(tA.q, -d));
    nv.wA = xmul(tA, pA.vertex(nv.indexA));
    nv.indexB = pB.support(rmulT(tB.q, d));
    nv.wB = xmul(tB, pB.vertex(nv.indexB));
    nv.w = nv.wB - nv.wA;
    nv.a = 0.0f;
    ++iter;
    const bool duplicate = (saveCount > 0 && nv.indexA == sA0 && nv.indexB == sB0) ||
                           (saveCount > 1 && nv.indexA == sA1 && nv.indexB == sB1) ||
                           (saveCount > 2 && nv.indexA == sA2 && nv.indexB == sB2);
    if (duplicate) break;
    if (count == 1) v1 = nv;
    else v2 = nv;
    ++count;
  }
  V2 pointA, pointB;
  if (count == 1) {
    pointA = v0.wA;
    pointB = v0.wB;
  } else if (count == 2) {
    pointA = v0.a * v0.wA + v1.a * v1.wA;
    pointB = v0.a * v0.wB + v1.a * v1.wB;
  } else {
    pointA = v0.a * v0.wA + v1.a * v1.wA + v2.a * v2.wA;
    pointB = pointA;
  }
  float distance = length(pointA - pointB);
  cache.metric = simplex_metric(count, v0, v1, v2);
  cache.count = count;
  cache.iA0 = v0.indexA; cache.iB0 = v0.indexB;
  cache.iA1 = v1.indexA; cache.iB1 = v1.indexB;
  cache.iA2 = v2.indexA; cache.iB2 = v2.indexB;
  return distance;
}

// b2SeparationFunction
template <class PA, class PB>
struct SepFn {
  PA pA;
  PB pB;
  SweepD sA, sB;
  int type;  // 0 points, 1 faceA, 2 faceB
  V2 localPoint, axis;

  __device__ __forceinline__ void initialize(const SimplexCache& cache, const PA& a, const SweepD& sa, const PB& b,
                                             const SweepD& sb, float t1) {
    pA = a;
    pB = b;
    sA = sa;
    sB = sb;
    localPoint = mk(0.0f, 0.0f);
    Xf xfA = sweep_xf(sA, t1), xfB = sweep_xf(sB, t1);
    if (cache.count == 1) {
      type = 0;
      V2 pointA = xmul(xfA, pA.vertex(cache.iA0));
      V2 pointB = xmul(xfB, pB.vertex(cache.iB0));
      axis = pointB - pointA;
      normalize(axis);
    } else if (cache.iA0 == cache.iA1) {
      type = 2;
      V2 localPointB1 = pB.vertex(cache.iB0);
      V2 localPointB2 = pB.vertex(cache.iB1);
      axis = cross(localPointB2 - localPointB1, 1.0f);
      normalize(axis);
      V2 normal = rmul(xfB.q, axis);
      localPoint = 0.5f * (localPointB1 + localPointB2);
      V2 pointB = xmul(xfB, localPoint);
      V2 pointA = xmul(xfA, pA.vertex(cache.iA0));
      float s = dot(pointA - pointB, normal);
      if (s < 0.0f) axis = -axis;
    } else {
      type = 1;
      V2 localPointA1 = pA.vertex(cache.iA0);
      V2 localPointA2 = pA.vertex(cache.iA1);
      axis = cross(localPointA2 - localPointA1, 1.0f);
      normalize(axis);
      V2 normal = rmul(xfA.q, axis);
      localPoint = 0.5f * (localPointA1 + localPointA2);
      V2 pointA = xmul(xfA, localPoint);
      V2 pointB = xmul(xfB, pB.vertex(cache.iB0));
      float s = dot(pointB - pointA, normal);
      if (s < 0.0f) axis = -axis;
    }
  }
  __device__ __forceinline__ float findMinSeparation(int& indexA, int& indexB, float t) const {
    Xf xfA = sweep_xf(sA, t), xfB = sweep_xf(sB, t);
    if (type == 0) {
      V2 axisA = rmulT(xfA.q, axis);
      V2 axisB = rmulT(xfB.q, -axis);
      indexA = pA.support(axisA);
      indexB = pB.support(axisB);
      V2 pointA = xmul(xfA, pA.vertex(indexA));
      V2 pointB = xmul(xfB, pB.vertex(indexB));
      return dot(pointB - pointA, axis);
    } else if (type == 1) {
      V2 normal = rmul(xfA.q, axis);
      V2 pointA = xmul(xfA, localPoint);
      V2 axisB = rmulT(xfB.q, -normal);
      indexA = -1;
      indexB = pB.support(axisB);
      V2 pointB = xmul(xfB, pB.vertex(indexB));
      return dot(pointB - pointA, normal);
    } else {
      V2 normal = rmul(xfB.q, axis);
      V2 pointB = xmul(xfB, localPoint);
      V2 axisA = rmulT(xfA.q, -normal);
      indexB = -1;
      indexA = pA.support(axisA);
      V2 pointA = xmul(xfA, pA.vertex(indexA));
      return dot(pointA - pointB, normal);
    }
  }
  __device__ __forceinline__ float evaluate(int indexA, int indexB, float t) const {
    Xf xfA = sweep_xf(sA, t), xfB = sweep_xf(sB, t);
    if (type == 0) {
      V2 pointA = xmul(xfA, pA.vertex(indexA));
      V2 pointB = xmul(xfB, pB.vertex(indexB));
      return dot(pointB - pointA, axis);
    } else if (type == 1) {
      V2 normal = rmul(xfA.q, axis);
      V2 pointA = xmul(xfA, localPoint);
      V2 pointB = xmul(xfB, pB.vertex(indexB));
      return dot(pointB - pointA, normal);
    } else {
      V2 normal = rmul(xfB.q, axis);
      V2 pointB = xmul(xfB, localPoint);
      V2 pointA = xmul(xfA, pA.vertex(indexA));
      return dot(pointA - pointB, normal);
    }
  }
};

// b2TimeOfImpact with tMax = 1.  Returns t >= 0 if the state is e_touching, a negative value otherwise.
template <class PA, class PB>
__device__ __forceinline__ float time_of_impact_t(const ProxyConst* shapeA, SweepD sweepA, const ProxyConst* shapeB,
                                                  SweepD sweepB) {
  PA proxyA;
  PB proxyB;
  proxyA.set(shapeA);
  proxyB.set(shapeB);
  sweep_normalize(sweepA);
  sweep_normalize(sweepB);
  const float tMax = 1.0f;
  float totalRadius = proxyA.radius + proxyB.radius;
  float target = b2max(KB_LINEAR_SLOP, totalRadius - 3.0f * KB_LINEAR_SLOP);
  float tolerance = 0.25f * KB_LINEAR_SLOP;
  float t1 = 0.0f;
  const int k_maxIterations = 20;
  int iter = 0;
  SimplexCache cache;
  cache.metric = 0.0f;
  cache.count = 0;
  cache.iA0 = cache.iA1 = cache.iA2 = cache.iB0 = cache.iB1 = cache.iB2 = 0;
  for (;;) {
    Xf xfA = sweep_xf(sweepA, t1), xfB = sweep_xf(sweepB, t1);
    float distance = gjk_distance(cache, proxyA, xfA, proxyB, xfB);
    if (distance <= 0.0f) return -1.0f;  // e_overlapped
    if (distance < target + tolerance) return t1;  // e_touching
    SepFn<PA, PB> fcn;
    fcn.initialize(cache, proxyA, sweepA, proxyB, sweepB, t1);
    bool done = false;
    float t2 = tMax;
    int pushBackIter = 0;
    for (;;) {
      int indexA, indexB;
      float s2 = fcn.findMinSeparation(indexA, indexB, t2);
      if (s2 > target + tolerance) return -1.0f;  // e_separated
      if (s2 > target - tolerance) {
        t1 = t2;
        break;
      }
      float s1 = fcn.evaluate(indexA, indexB, t1);
      if (s1 < target - tolerance) return -1.0f;  // e_failed
      if (s1 <= target + tolerance) return t1;  // e_touching
      int rootIterCount = 0;
      float a1 = t1, a2 = t2;
      for (;;) {
        float t;
        if (rootIterCount & 1) t = a1 + (target - s1) * (a2 - a1) / (s2 - s1);
        else t = 0.5f * (a1 + a2);
        ++rootIterCount;
        float s = fcn.evaluate(indexA, indexB, t);
        if (b2abs(s - target) < tolerance) {
          t2 = t;
          break;
        }
        if (s > target) {
          a1 = t;
          s1 = s;
        } else {
          a2 = t;
          s2 = s;
        }
        if (rootIterCount == 50) break;
      }
      ++pushBackIter;
      if (pushBackIter == KB_MAX_POLY_VERTS) break;
    }
    ++iter;
    if (done) break;
    if (iter == k_maxIterations) return -1.0f;  // e_failed
  }
  return -1.0f;
}

__device__ __noinline__ float time_of_impact(const ProxyConst* shapeA, SweepD sweepA, const ProxyConst* shapeB,
                                             SweepD sweepB) {
  return time_of_impact_t<DProxy, DProxy>(shapeA, sweepA, shapeB, sweepB);
}
// table edge against a circle (a kilobot or a Circle object)
__device__ __noinline__ float time_of_impact_edge_circle(const ProxyConst* shapeA, SweepD sweepA, const ProxyConst* shapeB,
                                                         SweepD sweepB) {
  return time_of_impact_t<DProxyEdge, DProxyCircle>(shapeA, sweepA, shapeB, sweepB);
}

// ------------------------------------------------------------------------ b2World::SolveTOI
template <int LPE, bool UNI, class LT>
__device__ __noinline__ uint32_t solveTOINI(Sim<LPE, UNI, LT> s) {
  const uint32_t before = s.nToi;
  s.solveTOI();
  return s.nToi - before;
}

// (the caller has already established that at least one contact with the table exists)
template <int LPE, bool UNI, class LT>
__device__ __forceinline__ void Sim<LPE, UNI, LT>::solveTOI() {
  const int B = L.B;
  int nC = (int)hdr(H_NC);

  for (int b = g.lane; b <= B; b += LPE) sweep4(b).set(3, 0.0f);  // alpha0 = 0
  for (int i = g.lane; i < nC; i += LPE) {
    cw(i) &= ~(CI_TOI | CI_TOICOUNT_MASK);
    toiAlpha(i) = f2u(1.0f);
  }
  g.sync();

  for (int guard = 0; guard < 64 * KB_MAX_SUB_STEPS; ++guard) {
#ifdef KB_PROFILE
    long long tq0 = clock64();
    if (profOut && g.lane == 0) profOut[15] += 1ull;   // rounds
#endif
    nC = (int)hdr(H_NC);
    const float tableAlpha0 = sweep4(S).get(3);
    // ---- per-contact TOI (lane parallel).  Bodies lagging behind the table's alpha0 are
    //      advanced first (b2Sweep::Advance is idempotent for a common target).
    for (int base = 0; base < nC; base += LPE) {
      const int i = base + g.lane;
      bool need = false;
      int pa = 0, pb = 0, bd = S;
      if (i < nC) {
        const uint32_t w = cw(i);
        const bool enabled = (w & CI_ENABLED) != 0u;
        const int toiCount = (w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT;
        if (enabled && toiCount <= KB_MAX_SUB_STEPS && (w & CI_TOI) == 0u) {
          pa = CW_PA(w);
          pb = CW_PB(w);
          const int bA = pbody(pa), bB = pbody(pb);
          // chain is always fixture A, so the table can only be body A
          if (bA == S && bB != S && awake(bB)) {
            need = true;
            bd = bB;
          }
        }
      }
      if (need) {
        float4 sw = sweep4(bd);
        if (sw.w < tableAlpha0) {
          // b2Sweep::Advance(alpha0)
          const float4 p = pos4(bd);
          float beta = (tableAlpha0 - sw.w) / (1.0f - sw.w);
          sw.x += beta * (p.x - sw.x);
          sw.y += beta * (p.y - sw.y);
          sw.z += beta * (p.z - sw.z);
          sw.w = tableAlpha0;
          sweep4(bd) = sw;
        }
      }
      g.sync();
      if (need) {
        const float4 sw = sweep4(bd);
        const float4 p = pos4(bd);
        const float4 k = bc4(bd);
        SweepD sA, sB;
        sA.lc = mk(0.0f, 0.0f); sA.c0 = mk(0.0f, 0.0f); sA.c = mk(0.0f, 0.0f);
        sA.a0 = 0.0f; sA.a = 0.0f; sA.alpha0 = tableAlpha0;
        sA.fixedRot = 1;
        sB.lc = mk(k.z, k.w); sB.c0 = mk(sw.x, sw.y); sB.c = mk(p.x, p.y);
        sB.a0 = sw.z; sB.a = p.z; sB.alpha0 = sw.w;
        sB.fixedRot = (ptype(pb) == SHAPE_CIRCLE && k.z == 0.0f && k.w == 0.0f) ? 1 : 0;
        const float alpha0 = tableAlpha0;
        float alpha = 1.0f;
        {
          const float t = (ptype(pa) == SHAPE_EDGE && ptype(pb) == SHAPE_CIRCLE)
                              ? time_of_impact_edge_circle(px + pa, sA, px + pb, sB)
                              : time_of_impact(px + pa, sA, px + pb, sB);
          if (t >= 0.0f) alpha = b2min(alpha0 + (1.0f - alpha0) * t, 1.0f);
        }
        toiAlpha(i) = f2u(alpha);
        cw(i) |= CI_TOI;
      }
      g.sync();
    }
#ifdef KB_PROFILE
    if (profOut && g.lane == 0) profOut[13] += (unsigned long long)(clock64() - tq0);   // TOI computations
    tq0 = clock64();
#endif
    // ---- minimum alpha, first in world-list order (highest index) on ties
    uint32_t bestBits = f2u(1.0f);
    int bestIdx = -1;
    for (int base = 0; base < nC; base += LPE) {
      const int i = base + g.lane;
      if (i < nC) {
        const uint32_t w = cw(i);
        const int toiCount = (w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT;
        if ((w & CI_ENABLED) != 0u && toiCount <= KB_MAX_SUB_STEPS && (w & CI_TOI) != 0u) {
          const float alpha = u2f(toiAlpha(i));
          if (alpha < 1.0f) {
            const uint32_t bits = f2u(alpha);
            if (bits < bestBits || (bits == bestBits && i > bestIdx)) {
              bestBits = bits;
              bestIdx = i;
            }
          }
        }
      }
    }
    const uint32_t minBits = __reduce_min_sync(g.gmask, bestBits);
    const int cand = (bestBits == minBits && bestIdx >= 0) ? bestIdx : -1;
    const int minContact = (int)__reduce_max_sync(g.gmask, (uint32_t)(cand + 1)) - 1;
    const float minAlpha = u2f(minBits);
    if (minContact < 0 || 1.0f - 10.0f * KB_EPS < minAlpha) break;

    nToi += 1u;
    const int bd = pbody(CW_PB(cw(minContact)));  // the dynamic body (fixture B)
    // backups, advance both bodies to minAlpha (b2Body::Advance)
    const float4 backupSweep = sweep4(bd), backupPos = pos4(bd), backupXf = xf4(bd);
    const float4 backupTable = sweep4(S);
    g.sync();
    if (g.lane == 0) {
      float4 sw = sweep4(bd);
      float4 p = pos4(bd);
      const float4 k = bc4(bd);
      float beta = (minAlpha - sw.w) / (1.0f - sw.w);
      sw.x += beta * (p.x - sw.x);
      sw.y += beta * (p.y - sw.y);
      sw.z += beta * (p.z - sw.z);
      sw.w = minAlpha;
      p.x = sw.x; p.y = sw.y; p.z = sw.z;
      sweep4(bd) = sw;
      pos4(bd) = p;
      Rot q = rot_set(p.z);
      V2 o = mk(p.x, p.y) - rmul(q, mk(k.z, k.w));
      xf4(bd) = make_float4(o.x, o.y, q.s, q.c);
      sweep4(S).set(3, minAlpha);
      // minContact->Update()
      updateContact(minContact);
      uint32_t w = cw(minContact);
      w &= ~CI_TOI;
      const uint32_t tc = ((w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT) + 1u;
      w = (w & ~CI_TOICOUNT_MASK) | (tc << CI_TOICOUNT_SHIFT);
      cw(minContact) = w;
    }
    g.sync();
    if ((cw(minContact) & CI_TOUCHING) == 0u) {
      g.sync();
      if (g.lane == 0) {
        cw(minContact) &= ~CI_ENABLED;
        sweep4(bd) = backupSweep;
        // restoring m_sweep leaves c/a at the backup values; SynchronizeTransform
        pos4(bd) = backupPos;
        xf4(bd) = backupXf;
        sweep4(S) = backupTable;
      }
      g.sync();
      continue;
    }
    if (g.lane == 0) wake(bd);
    g.sync();
    // ---- mini island: minContact first, then the body's other touching wall contacts in list order
    //      (each re-evaluated at the advanced pose)
    const int islandCap = min(KB_MAX_TOI_CONTACTS, min(L.Gmax, L.Kmax));
    {
      // records of the mini island: behind the TOI cache in the record region if they fit, else in the blob
      const int first = 3 * L.Kmax + 8 + L.Cmax;
      genBase = (first + GR_WORDS * islandCap <= L.recWords) ? smemGeneric(L.sRec + first) : blob + L.oGen;
    }
    int nIsland = 1;
    if (g.lane == 0) ord(0) = (uint32_t)minContact;
    for (int base = 0; base < nC; base += LPE) {
      const int i = nC - 1 - (base + g.lane);
      bool add = false;
      if (i >= 0 && i != minContact) {
        const uint32_t w = cw(i);
        if (pbody(CW_PA(w)) == S && pbody(CW_PB(w)) == bd) {
          updateContact(i);
          add = (cw(i) & (CI_ENABLED | CI_TOUCHING)) == (CI_ENABLED | CI_TOUCHING);
        }
      }
      const uint32_t m = g.ballot(add);
      const int dst = nIsland + __popc(m & g.lt());
      if (add && dst < islandCap) ord(dst) = (uint32_t)i;
      nIsland = min(nIsland + __popc(m), islandCap);
    }
    g.sync();
    // ---- b2Island::SolveTOI (one dynamic body: strictly sequential, lane 0; general-constraint records)
    if (g.lane == 0) {
      const float subDt = (1.0f - minAlpha) * L.dt;
      // position constraints first: load manifold data into the records (position layout)
      for (int k = 0; k < nIsland; ++k) {
        const int ci = (int)ord(k);
        const uint32_t tp = f2u(manifoldRec(ci)[MR_TYPE]);
        const uint32_t type = tp & 0xFF, pointCount = (tp >> 8) & 0xFF;
        poolu(PF_IDX, k) = (uint32_t)S | ((uint32_t)bd << 8) | (pointCount << 16) | (type << 24) | (pointCount << 28);
        poolu(PF_AUX, k) = (uint32_t)ci;
        preparePositionGeneral(k, ci);
      }
      for (int it = 0; it < 20; ++it) {
        bool ok = true;
        for (int k = 0; k < nIsland; ++k) ok &= solvePositionGeneral(k, KB_TOI_BAUMGARTE, -1.5f * KB_LINEAR_SLOP, S, bd);
        if (ok) break;
      }
      {
        const float4 p = pos4(bd);
        sweep4(bd).set(0, p.x); sweep4(bd).set(1, p.y); sweep4(bd).set(2, p.z);  // c0, a0 = corrected pose
      }
      // velocity constraints without warm starting, at the corrected pose
      for (int k = 0; k < nIsland; ++k) initGeneral(k, (int)ord(k), S, bd, ord(k), true);
      for (int it = 0; it < L.velIters; ++it)
        for (int k = 0; k < nIsland; ++k) solveVelocityGeneral(k);
      // integrate the remainder of the step
      {
        const float h = subDt;
        float4 p = pos4(bd);
        float4 v = vel4(bd);
        const float4 kk = bc4(bd);
        V2 translation = h * mk(v.x, v.y);
        if (dot(translation, translation) > KB_MAX_TRANSLATION_SQ) {
          float ratio = KB_MAX_TRANSLATION / length(translation);
          v.x *= ratio;
          v.y *= ratio;
        }
        float rotation = h * v.z;
        if (rotation * rotation > KB_MAX_ROTATION_SQ) {
          float ratio = KB_MAX_ROTATION / b2abs(rotation);
          v.z *= ratio;
        }
        p.x += h * v.x;
        p.y += h * v.y;
        p.z += h * v.z;
        pos4(bd) = p;
        vel4(bd) = v;
        Rot q = rot_set(p.z);
        V2 o = mk(p.x, p.y) - rmul(q, mk(kk.z, kk.w));
        xf4(bd) = make_float4(o.x, o.y, q.s, q.c);
      }
      for (int b = 0; b <= B; ++b) isl(b) = b == bd ? 0 : -1;
    }
    g.sync();
    synchronizeFixtures(true);
    // invalidate the cached TOIs of every contact of the displaced body
    for (int i = g.lane; i < nC; i += LPE) {
      const uint32_t w = cw(i);
      if (pbody(CW_PA(w)) == bd || pbody(CW_PB(w)) == bd) cw(i) = w & ~CI_TOI;
    }
    g.sync();
    const int before = (int)hdr(H_NC);
    findNewContacts();
    const int after = (int)hdr(H_NC);
    for (int i = before + g.lane; i < after; i += LPE) toiAlpha(i) = f2u(1.0f);
    g.sync();
#ifdef KB_PROFILE
    if (profOut && g.lane == 0) profOut[14] += (unsigned long long)(clock64() - tq0);   // event handling
#endif
  }
}

}  // namespace kb
