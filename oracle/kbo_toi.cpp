// CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED (see kbo_math.h).
// Restates b2Distance.cpp (GJK with simplex cache) and b2TimeOfImpact.cpp (conservative
// advancement with b2SeparationFunction) of Box2D 2.3.x -- SURVEY.md Appendix B.8.  Reached from
// b2World::SolveTOI for dynamic-vs-static (table) contacts only.
#include "kbo_world.h"

namespace kbo {
namespace {

struct DistanceProxy {
  Vec2 buffer[kMaxPolygonVertices];
  const Vec2* vertices;
  int count;
  float radius;
  void Set(const Shape* shape) {
    switch (shape->type) {
      case kCircle:
        buffer[0] = shape->p;
        vertices = buffer;
        count = 1;
        radius = shape->radius;
        break;
      case kPolygon:
        vertices = shape->vertices;
        count = shape->count;
        radius = shape->radius;
        break;
      default:  // chain child edge
        buffer[0] = shape->v1;
        buffer[1] = shape->v2;
        vertices = buffer;
        count = 2;
        radius = shape->radius;
        break;
    }
  }
  int GetSupport(const Vec2& d) const {
    int bestIndex = 0;
    float bestValue = Dot(vertices[0], d);
    for (int i = 1; i < count; ++i) {
      float value = Dot(vertices[i], d);
      if (value > bestValue) {
        bestIndex = i;
        bestValue = value;
      }
    }
    return bestIndex;
  }
  const Vec2& GetVertex(int index) const { return vertices[index]; }
};

struct SimplexCache {
  float metric;
  uint16_t count;
  uint8_t indexA[3];
  uint8_t indexB[3];
};

struct SimplexVertex {
  Vec2 wA, wB, w;
  float a;
  int indexA, indexB;
};

struct Simplex {
  SimplexVertex m_v[3];
  int m_count;

  float GetMetric() const {
    switch (m_count) {
      case 1: return 0.0f;
      case 2: return (m_v[0].w - m_v[1].w).Length();
      case 3: return Cross(m_v[1].w - m_v[0].w, m_v[2].w - m_v[0].w);
      default: return 0.0f;
    }
  }
  void ReadCache(const SimplexCache* cache, const DistanceProxy* proxyA, const Xf& transformA,
                 const DistanceProxy* proxyB, const Xf& transformB) {
    m_count = cache->count;
    for (int i = 0; i < m_count; ++i) {
      SimplexVertex* v = m_v + i;
      v->indexA = cache->indexA[i];
      v->indexB = cache->indexB[i];
      Vec2 wALocal = proxyA->GetVertex(v->indexA);
      Vec2 wBLocal = proxyB->GetVertex(v->indexB);
      v->wA = Mul(transformA, wALocal);
      v->wB = Mul(transformB, wBLocal);
      v->w = v->wB - v->wA;
      v->a = 0.0f;
    }
    if (m_count > 1) {
      float metric1 = cache->metric;
      float metric2 = GetMetric();
      if (metric2 < 0.5f * metric1 || 2.0f * metric1 < metric2 || metric2 < kEpsilon) m_count = 0;
    }
    if (m_count == 0) {
      SimplexVertex* v = m_v + 0;
      v->indexA = 0;
      v->indexB = 0;
      Vec2 wALocal = proxyA->GetVertex(0);
      Vec2 wBLocal = proxyB->GetVertex(0);
      v->wA = Mul(transformA, wALocal);
      v->wB = Mul(transformB, wBLocal);
      v->w = v->wB - v->wA;
      v->a = 1.0f;
      m_count = 1;
    }
  }
  void WriteCache(SimplexCache* cache) const {
    cache->metric = GetMetric();
    cache->count = (uint16_t)m_count;
    for (int i = 0; i < m_count; ++i) {
      cache->indexA[i] = (uint8_t)m_v[i].indexA;
      cache->indexB[i] = (uint8_t)m_v[i].indexB;
    }
  }
  Vec2 GetSearchDirection() const {
    switch (m_count) {
      case 1: return -m_v[0].w;
      case 2: {
        Vec2 e12 = m_v[1].w - m_v[0].w;
        float sgn = Cross(e12, -m_v[0].w);
        if (sgn > 0.0f) return Cross(1.0f, e12);
        return Cross(e12, 1.0f);
      }
      default: return Vec2(0.0f, 0.0f);
    }
  }
  Vec2 GetClosestPoint() const {
    switch (m_count) {
      case 1: return m_v[0].w;
      case 2: return m_v[0].a * m_v[0].w + m_v[1].a * m_v[1].w;
      default: return Vec2(0.0f, 0.0f);
    }
  }
  void GetWitnessPoints(Vec2* pA, Vec2* pB) const {
    switch (m_count) {
      case 1:
        *pA = m_v[0].wA;
        *pB = m_v[0].wB;
        break;
      case 2:
        *pA = m_v[0].a * m_v[0].wA + m_v[1].a * m_v[1].wA;
        *pB = m_v[0].a * m_v[0].wB + m_v[1].a * m_v[1].wB;
        break;
      case 3:
        *pA = m_v[0].a * m_v[0].wA + m_v[1].a * m_v[1].wA + m_v[2].a * m_v[2].wA;
        *pB = *pA;
        break;
      default: break;
    }
  }
  void Solve2() {
    Vec2 w1 = m_v[0].w;
    Vec2 w2 = m_v[1].w;
    Vec2 e12 = w2 - w1;
    float d12_2 = -Dot(w1, e12);
    if (d12_2 <= 0.0f) {
      m_v[0].a = 1.0f;
      m_count = 1;
      return;
    }
    float d12_1 = Dot(w2, e12);
    if (d12_1 <= 0.0f) {
      m_v[1].a = 1.0f;
      m_count = 1;
      m_v[0] = m_v[1];
      return;
    }
    float inv_d12 = 1.0f / (d12_1 + d12_2);
    m_v[0].a = d12_1 * inv_d12;
    m_v[1].a = d12_2 * inv_d12;
    m_count = 2;
  }
  void Solve3() {
    Vec2 w1 = m_v[0].w;
    Vec2 w2 = m_v[1].w;
    Vec2 w3 = m_v[2].w;
    Vec2 e12 = w2 - w1;
    float w1e12 = Dot(w1, e12);
    float w2e12 = Dot(w2, e12);
    float d12_1 = w2e12;
    float d12_2 = -w1e12;
    Vec2 e13 = w3 - w1;
    float w1e13 = Dot(w1, e13);
    float w3e13 = Dot(w3, e13);
    float d13_1 = w3e13;
    float d13_2 = -w1e13;
    Vec2 e23 = w3 - w2;
    float w2e23 = Dot(w2, e23);
    float w3e23 = Dot(w3, e23);
    float d23_1 = w3e23;
    float d23_2 = -w2e23;
    float n123 = Cross(e12, e13);
    float d123_1 = n123 * Cross(w2, w3);
    float d123_2 = n123 * Cross(w3, w1);
    float d123_3 = n123 * Cross(w1, w2);
    if (d12_2 <= 0.0f && d13_2 <= 0.0f) {
      m_v[0].a = 1.0f;
      m_count = 1;
      return;
    }
    if (d12_1 > 0.0f && d12_2 > 0.0f && d123_3 <= 0.0f) {
      float inv_d12 = 1.0f / (d12_1 + d12_2);
      m_v[0].a = d12_1 * inv_d12;
      m_v[1].a = d12_2 * inv_d12;
      m_count = 2;
      return;
    }
    if (d13_1 > 0.0f && d13_2 > 0.0f && d123_2 <= 0.0f) {
      float inv_d13 = 1.0f / (d13_1 + d13_2);
      m_v[0].a = d13_1 * inv_d13;
      m_v[2].a = d13_2 * inv_d13;
      m_count = 2;
      m_v[1] = m_v[2];
      return;
    }
    if (d12_1 <= 0.0f && d23_2 <= 0.0f) {
      m_v[1].a = 1.0f;
      m_count = 1;
      m_v[0] = m_v[1];
      return;
    }
    if (d13_1 <= 0.0f && d23_1 <= 0.0f) {
      m_v[2].a = 1.0f;
      m_count = 1;
      m_v[0] = m_v[2];
      return;
    }
    if (d23_1 > 0.0f && d23_2 > 0.0f && d123_1 <= 0.0f) {
      float inv_d23 = 1.0f / (d23_1 + d23_2);
      m_v[1].a = d23_1 * inv_d23;
      m_v[2].a = d23_2 * inv_d23;
      m_count = 2;
      m_v[0] = m_v[2];
      return;
    }
    float inv_d123 = 1.0f / (d123_1 + d123_2 + d123_3);
    m_v[0].a = d123_1 * inv_d123;
    m_v[1].a = d123_2 * inv_d123;
    m_v[2].a = d123_3 * inv_d123;
    m_count = 3;
  }
};

// b2Distance with useRadii = false; returns the distance between the core shapes.
float Distance(SimplexCache* cache, const DistanceProxy* proxyA, const Xf& transformA,
               const DistanceProxy* proxyB, const Xf& transformB) {
  Simplex simplex;
  simplex.ReadCache(cache, proxyA, transformA, proxyB, transformB);
  SimplexVertex* vertices = simplex.m_v;
  const int k_maxIters = 20;
  int saveA[3], saveB[3];
  int saveCount = 0;
  int iter = 0;
  while (iter < k_maxIters) {
    saveCount = simplex.m_count;
    for (int i = 0; i < saveCount; ++i) {
      saveA[i] = vertices[i].indexA;
      saveB[i] = vertices[i].indexB;
    }
    switch (simplex.m_count) {
      case 1: break;
      case 2: simplex.Solve2(); break;
      case 3: simplex.Solve3(); break;
    }
    if (simplex.m_count == 3) break;
    Vec2 d = simplex.GetSearchDirection();
    if (d.LengthSquared() < kEpsilon * kEpsilon) break;
    SimplexVertex* vertex = vertices + simplex.m_count;
    vertex->indexA = proxyA->GetSupport(MulT(transformA.q, -d));
    vertex->wA = Mul(transformA, proxyA->GetVertex(vertex->indexA));
    vertex->indexB = proxyB->GetSupport(MulT(transformB.q, d));
    vertex->wB = Mul(transformB, proxyB->GetVertex(vertex->indexB));
    vertex->w = vertex->wB - vertex->wA;
    ++iter;
    bool duplicate = false;
    for (int i = 0; i < saveCount; ++i) {
      if (vertex->indexA == saveA[i] && vertex->indexB == saveB[i]) {
        duplicate = true;
        break;
      }
    }
    if (duplicate) break;
    ++simplex.m_count;
  }
  Vec2 pointA, pointB;
  simplex.GetWitnessPoints(&pointA, &pointB);
  float distance = (pointA - pointB).Length();
  simplex.WriteCache(cache);
  return distance;
}

struct SeparationFunction {
  enum Type { kPoints, kFaceA, kFaceB };
  const DistanceProxy* m_proxyA;
  const DistanceProxy* m_proxyB;
  Sweep m_sweepA, m_sweepB;
  Type m_type;
  Vec2 m_localPoint;
  Vec2 m_axis;

  float Initialize(const SimplexCache* cache, const DistanceProxy* proxyA, const Sweep& sweepA,
                   const DistanceProxy* proxyB, const Sweep& sweepB, float t1) {
    m_proxyA = proxyA;
    m_proxyB = proxyB;
    int count = cache->count;
    m_sweepA = sweepA;
    m_sweepB = sweepB;
    Xf xfA, xfB;
    m_sweepA.GetTransform(&xfA, t1);
    m_sweepB.GetTransform(&xfB, t1);
    if (count == 1) {
      m_type = kPoints;
      Vec2 localPointA = m_proxyA->GetVertex(cache->indexA[0]);
      Vec2 localPointB = m_proxyB->GetVertex(cache->indexB[0]);
      Vec2 pointA = Mul(xfA, localPointA);
      Vec2 pointB = Mul(xfB, localPointB);
      m_axis = pointB - pointA;
      float s = m_axis.Normalize();
      return s;
    } else if (cache->indexA[0] == cache->indexA[1]) {
      m_type = kFaceB;
      Vec2 localPointB1 = proxyB->GetVertex(cache->indexB[0]);
      Vec2 localPointB2 = proxyB->GetVertex(cache->indexB[1]);
      m_axis = Cross(localPointB2 - localPointB1, 1.0f);
      m_axis.Normalize();
      Vec2 normal = Mul(xfB.q, m_axis);
      m_localPoint = 0.5f * (localPointB1 + localPointB2);
      Vec2 pointB = Mul(xfB, m_localPoint);
      Vec2 localPointA = proxyA->GetVertex(cache->indexA[0]);
      Vec2 pointA = Mul(xfA, localPointA);
      float s = Dot(pointA - pointB, normal);
      if (s < 0.0f) {
        m_axis = -m_axis;
        s = -s;
      }
      return s;
    } else {
      m_type = kFaceA;
      Vec2 localPointA1 = m_proxyA->GetVertex(cache->indexA[0]);
      Vec2 localPointA2 = m_proxyA->GetVertex(cache->indexA[1]);
      m_axis = Cross(localPointA2 - localPointA1, 1.0f);
      m_axis.Normalize();
      Vec2 normal = Mul(xfA.q, m_axis);
      m_localPoint = 0.5f * (localPointA1 + localPointA2);
      Vec2 pointA = Mul(xfA, m_localPoint);
      Vec2 localPointB = m_proxyB->GetVertex(cache->indexB[0]);
      Vec2 pointB = Mul(xfB, localPointB);
      float s = Dot(pointB - pointA, normal);
      if (s < 0.0f) {
        m_axis = -m_axis;
        s = -s;
      }
      return s;
    }
  }

  float FindMinSeparation(int* indexA, int* indexB, float t) const {
    Xf xfA, xfB;
    m_sweepA.GetTransform(&xfA, t);
    m_sweepB.GetTransform(&xfB, t);
    switch (m_type) {
      case kPoints: {
        Vec2 axisA = MulT(xfA.q, m_axis);
        Vec2 axisB = MulT(xfB.q, -m_axis);
        *indexA = m_proxyA->GetSupport(axisA);
        *indexB = m_proxyB->GetSupport(axisB);
        Vec2 localPointA = m_proxyA->GetVertex(*indexA);
        Vec2 localPointB = m_proxyB->GetVertex(*indexB);
        Vec2 pointA = Mul(xfA, localPointA);
        Vec2 pointB = Mul(xfB, localPointB);
        return Dot(pointB - pointA, m_axis);
      }
      case kFaceA: {
        Vec2 normal = Mul(xfA.q, m_axis);
        Vec2 pointA = Mul(xfA, m_localPoint);
        Vec2 axisB = MulT(xfB.q, -normal);
        *indexA = -1;
        *indexB = m_proxyB->GetSupport(axisB);
        Vec2 localPointB = m_proxyB->GetVertex(*indexB);
        Vec2 pointB = Mul(xfB, localPointB);
        return Dot(pointB - pointA, normal);
      }
      default: {
        Vec2 normal = Mul(xfB.q, m_axis);
        Vec2 pointB = Mul(xfB, m_localPoint);
        Vec2 axisA = MulT(xfA.q, -normal);
        *indexB = -1;
        *indexA = m_proxyA->GetSupport(axisA);
        Vec2 localPointA = m_proxyA->GetVertex(*indexA);
        Vec2 pointA = Mul(xfA, localPointA);
        return Dot(pointA - pointB, normal);
      }
    }
  }

  float Evaluate(int indexA, int indexB, float t) const {
    Xf xfA, xfB;
    m_sweepA.GetTransform(&xfA, t);
    m_sweepB.GetTransform(&xfB, t);
    switch (m_type) {
      case kPoints: {
        Vec2 localPointA = m_proxyA->GetVertex(indexA);
        Vec2 localPointB = m_proxyB->GetVertex(indexB);
        Vec2 pointA = Mul(xfA, localPointA);
        Vec2 pointB = Mul(xfB, localPointB);
        return Dot(pointB - pointA, m_axis);
      }
      case kFaceA: {
        Vec2 normal = Mul(xfA.q, m_axis);
        Vec2 pointA = Mul(xfA, m_localPoint);
        Vec2 localPointB = m_proxyB->GetVertex(indexB);
        Vec2 pointB = Mul(xfB, localPointB);
        return Dot(pointB - pointA, normal);
      }
      default: {
        Vec2 normal = Mul(xfB.q, m_axis);
        Vec2 pointB = Mul(xfB, m_localPoint);
        Vec2 localPointA = m_proxyA->GetVertex(indexA);
        Vec2 pointA = Mul(xfA, localPointA);
        return Dot(pointA - pointB, normal);
      }
    }
  }
};

}  // namespace

float DistanceCore(const Shape* shapeA, const Xf& xfA, const Shape* shapeB, const Xf& xfB, int* simplexCount) {
  DistanceProxy proxyA, proxyB;
  proxyA.Set(shapeA);
  proxyB.Set(shapeB);
  SimplexCache cache;
  cache.metric = 0.0f;
  cache.count = 0;
  const float d = Distance(&cache, &proxyA, xfA, &proxyB, xfB);
  *simplexCount = cache.count;
  return d;
}

void TimeOfImpact(TOIOutput* output, const TOIInput* input) {
  output->state = TOIOutput::kUnknown;
  output->t = input->tMax;
  DistanceProxy proxyA, proxyB;
  proxyA.Set(input->shapeA);
  proxyB.Set(input->shapeB);
  Sweep sweepA = input->sweepA;
  Sweep sweepB = input->sweepB;
  sweepA.Normalize();
  sweepB.Normalize();
  float tMax = input->tMax;
  float totalRadius = proxyA.radius + proxyB.radius;
  float target = Max(kLinearSlop, totalRadius - 3.0f * kLinearSlop);
  float tolerance = 0.25f * kLinearSlop;
  float t1 = 0.0f;
  const int k_maxIterations = 20;
  int iter = 0;
  SimplexCache cache;
  cache.metric = 0.0f;
  cache.count = 0;
  for (;;) {
    Xf xfA, xfB;
    sweepA.GetTransform(&xfA, t1);
    sweepB.GetTransform(&xfB, t1);
    float distance = Distance(&cache, &proxyA, xfA, &proxyB, xfB);
    if (distance <= 0.0f) {
      output->state = TOIOutput::kOverlapped;
      output->t = 0.0f;
      break;
    }
    if (distance < target + tolerance) {
      output->state = TOIOutput::kTouching;
      output->t = t1;
      break;
    }
    SeparationFunction fcn;
    fcn.Initialize(&cache, &proxyA, sweepA, &proxyB, sweepB, t1);
    bool done = false;
    float t2 = tMax;
    int pushBackIter = 0;
    for (;;) {
      int indexA, indexB;
      float s2 = fcn.FindMinSeparation(&indexA, &indexB, t2);
      if (s2 > target + tolerance) {
        output->state = TOIOutput::kSeparated;
        output->t = tMax;
        done = true;
        break;
      }
      if (s2 > target - tolerance) {
        t1 = t2;
        break;
      }
      float s1 = fcn.Evaluate(indexA, indexB, t1);
      if (s1 < target - tolerance) {
        output->state = TOIOutput::kFailed;
        output->t = t1;
        done = true;
        break;
      }
      if (s1 <= target + tolerance) {
        output->state = TOIOutput::kTouching;
        output->t = t1;
        done = true;
        break;
      }
      int rootIterCount = 0;
      float a1 = t1, a2 = t2;
      for (;;) {
        float t;
        if (rootIterCount & 1) t = a1 + (target - s1) * (a2 - a1) / (s2 - s1);
        else t = 0.5f * (a1 + a2);
        ++rootIterCount;
        float s = fcn.Evaluate(indexA, indexB, t);
        if (Abs(s - target) < tolerance) {
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
      if (pushBackIter == kMaxPolygonVertices) break;
    }
    ++iter;
    if (done) break;
    if (iter == k_maxIterations) {
      output->state = TOIOutput::kFailed;
      output->t = t1;
      break;
    }
  }
}

}  // namespace kbo
