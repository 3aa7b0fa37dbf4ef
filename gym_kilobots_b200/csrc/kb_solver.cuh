// kb_solver.cuh -- the contact-solver and island arithmetic that both kernel tiers run (kb_step.cuh / kb_toi.cuh, the
// lane-group tier, and kb_swarm.cuh, the large-swarm tier): functions on values, written once.  Every caller loads its
// operands from its own layout, calls one of these and stores the results itself, so the order of its shared-memory
// accesses stays its own and only the arithmetic is shared.
//
// The simple contact: one manifold point, no friction, no restitution, fixture B a circle at its body's origin (every
// contact of a kilobot).  Its velocity-phase records are v0 = (normal.x, normal.y, normalMass, normalImpulse) and
// v1 = (rA.x, rA.y, rB.x, rB.y); its position phase reads the manifold's (localNormal, localPoint).
#pragma once
#include "kb_types.cuh"

namespace kb {

// b2ContactSolver ctor + InitializeVelocityConstraints for a simple contact: b2WorldManifold::Initialize (e_circles /
// e_faceA) at the transforms (qA, cA - qA lcA) and (qB, cB - qB lcB), then the normal mass.  lnlp = (localNormal,
// localPoint) and mp = the local point of the manifold point; impulse is the warm-start impulse that goes into v0.w.
__device__ __forceinline__ void kb_init_simple(V2 cA, V2 cB, Rot qA, Rot qB, V2 lcA, V2 lcB, const float4& lnlp, V2 mp, int type,
                                               float radiusA, float radiusB, float mA, float iA, float mB, float iB, float impulse,
                                               float4& v0, float4& v1) {
  Xf xfA, xfB;
  xfA.q = qA;
  xfB.q = qB;
  xfA.p = cA - rmul(xfA.q, lcA);
  xfB.p = cB - rmul(xfB.q, lcB);
  V2 normal, pt;
  const V2 lp = mk(lnlp.z, lnlp.w), ln = mk(lnlp.x, lnlp.y);
  if (type == MANIFOLD_CIRCLES) {
    normal = mk(1.0f, 0.0f);
    V2 pointA = xmul(xfA, lp);
    V2 pointB = xmul(xfB, mp);
    if (distsq(pointA, pointB) > KB_EPS * KB_EPS) {
      normal = pointB - pointA;
      normalize(normal);
    }
    V2 a = pointA + radiusA * normal;
    V2 b = pointB - radiusB * normal;
    pt = 0.5f * (a + b);
  } else {
    normal = rmul(xfA.q, ln);
    V2 planePoint = xmul(xfA, lp);
    V2 clipPoint = xmul(xfB, mp);
    V2 a = clipPoint + (radiusA - dot(clipPoint - planePoint, normal)) * normal;
    V2 b = clipPoint - radiusB * normal;
    pt = 0.5f * (a + b);
  }
  const V2 rA = pt - cA;
  const V2 rB = pt - cB;
  const float rnA = cross(rA, normal);
  const float rnB = cross(rB, normal);
  const float kNormal = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
  const float nMass = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
  v0 = make_float4(normal.x, normal.y, nMass, impulse);
  v1 = make_float4(rA.x, rA.y, rB.x, rB.y);
}

// b2ContactSolver::WarmStart of a simple contact on the two bodies' (v.x, v.y, w, -) rows
__device__ __forceinline__ void kb_warm_start_simple(float4& vA, float4& vB, const float4& v0, const float4& v1, float mA, float iA,
                                                     float mB, float iB) {
  const V2 normal = mk(v0.x, v0.y);
  const V2 tangent = cross(normal, 1.0f);
  const V2 rA = mk(v1.x, v1.y), rB = mk(v1.z, v1.w);
  const V2 P = v0.w * normal + 0.0f * tangent;
  vA.z -= iA * cross(rA, P);
  vA.x = vA.x - mA * P.x;
  vA.y = vA.y - mA * P.y;
  vB.z += iB * cross(rB, P);
  vB.x = vB.x + mB * P.x;
  vB.y = vB.y + mB * P.y;
}

// b2ContactSolver::SolveVelocityConstraints of a simple contact (the tangent row contributes exactly zero: friction == 0).
// Returns the new accumulated normal impulse.
__device__ __forceinline__ float kb_solve_velocity_simple(float4& vA, float4& vB, const float4& v0, const float4& v1, float mA,
                                                          float iA, float mB, float iB) {
  const V2 normal = mk(v0.x, v0.y);
  const V2 rA0 = mk(v1.x, v1.y), rB0 = mk(v1.z, v1.w);
  const V2 Av = mk(vA.x, vA.y), Bv = mk(vB.x, vB.y);
  V2 dv = Bv + cross(vB.z, rB0) - Av - cross(vA.z, rA0);
  float vn = dot(dv, normal);
  float ni = v0.w;
  float lambda = -v0.z * (vn - 0.0f);
  float newImpulse = b2max(ni + lambda, 0.0f);
  lambda = newImpulse - ni;
  V2 P = lambda * normal;
  const V2 Av2 = Av - mA * P;
  vA.z -= iA * cross(rA0, P);
  const V2 Bv2 = Bv + mB * P;
  vB.z += iB * cross(rB0, P);
  vA.x = Av2.x; vA.y = Av2.y;
  vB.x = Bv2.x; vB.y = Bv2.y;
  return newImpulse;
}

// One constraint of b2ContactSolver::SolvePositionConstraints for a simple contact: b2PositionSolverManifold (e_circles /
// e_faceA) at the transforms (qA, cA - qA lcA) and (qB, cB - qB lcB), then the correction.  a0 / b0 = (c.x, c.y, angle, -)
// of the two bodies, a1 / b1 the corrected rows (only meaningful if `moved`).  Returns separation >= limit.
__device__ __forceinline__ bool kb_position_simple(const float4& a0, const float4& b0, Rot qA, Rot qB, V2 lcA, V2 lcB,
                                                   const float4& lnlp, int type, float radiusA, float radiusB, float mA, float iA,
                                                   float mB, float iB, float baumgarte, float limit, bool skipZero, float4& a1,
                                                   float4& b1, bool& moved) {
  V2 cA = mk(a0.x, a0.y), cB = mk(b0.x, b0.y);
  V2 normal, point;
  float separation;
  {
    const V2 ln = mk(lnlp.x, lnlp.y), lp = mk(lnlp.z, lnlp.w);
    Xf xfA, xfB;
    xfA.q = qA;
    xfB.q = qB;
    xfA.p = cA - rmul(xfA.q, lcA);
    xfB.p = cB - rmul(xfB.q, lcB);
    const V2 mpj = mk(0.0f, 0.0f);
    if (type == MANIFOLD_CIRCLES) {
      V2 pointA = xmul(xfA, lp);
      V2 pointB = xmul(xfB, mpj);
      normal = pointB - pointA;
      normalize(normal);
      point = 0.5f * (pointA + pointB);
      separation = dot(pointB - pointA, normal) - radiusA - radiusB;
    } else {
      normal = rmul(xfA.q, ln);
      V2 planePoint = xmul(xfA, lp);
      V2 clipPoint = xmul(xfB, mpj);
      separation = dot(clipPoint - planePoint, normal) - radiusA - radiusB;
      point = clipPoint;
    }
  }
  const bool ok = separation >= limit;
  const float C = b2clamp(baumgarte * (separation + KB_LINEAR_SLOP), -KB_MAX_LINEAR_CORRECTION, 0.0f);
  moved = false;
  if (skipZero && C == 0.0f) return ok;   // the impulse is -0 / K and moves nothing
  const V2 rA = point - cA;
  const V2 rB = point - cB;
  const float rnA = cross(rA, normal);
  const float rnB = cross(rB, normal);
  const float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
  const float impulse = K > 0.0f ? -C / K : 0.0f;
  const V2 P = impulse * normal;
  cA = cA - mA * P;
  const float aA = a0.z - iA * cross(rA, P);
  cB = cB + mB * P;
  const float aB = b0.z + iB * cross(rB, P);
  a1 = make_float4(cA.x, cA.y, aA, a0.w);
  b1 = make_float4(cB.x, cB.y, aB, b0.w);
  moved = true;
  return ok;
}

// One constraint of b2ContactSolver::SolvePositionConstraints for a circle-circle manifold whose local points and local
// centres are zero (kilobot against kilobot: xf.p == c, no rotation matters): the same operations in the same order as
// the general form, as straight-line code.  a0 / b0 = (c.x, c.y, angle, -) of the two bodies, a1 / b1 the corrected rows
// (only meaningful if `moved`).  EXACT_OPS: the plain operators; otherwise the *_u forms of kb_types.cuh (`bad` says
// whether the result may be used).
template <bool EXACT_OPS>
__device__ __forceinline__ bool kb_position_pair_t(const float4& a0, const float4& b0, float radiusA, float radiusB, float mA, float iA,
                                                   float mB, float iB, float baumgarte, float limit, bool skipZero, float4& a1,
                                                   float4& b1, bool& moved, bool& bad) {
  V2 cA = mk(a0.x, a0.y), cB = mk(b0.x, b0.y);
  V2 normal = cB - cA;
  if (EXACT_OPS) {
    normalize_plain(normal);
  } else {
    const float s = normal.x * normal.x + normal.y * normal.y;
    bad |= !KB_SQRT_WINDOW(s);
    const float len = kb_sqrt_raw(s);       // >= 2^-50.5 inside the window: the reciprocal needs no test of its own
    const float inv = kb_rcp_raw(len);
    const bool keep = len < KB_EPS;         // b2Vec2::Normalize leaves a vector shorter than epsilon alone
    normal.x = keep ? normal.x : normal.x * inv;
    normal.y = keep ? normal.y : normal.y * inv;
  }
  const V2 point = 0.5f * (cA + cB);
  const float separation = dot(cB - cA, normal) - radiusA - radiusB;
  const bool ok = separation >= limit;
  const float C = b2clamp(baumgarte * (separation + KB_LINEAR_SLOP), -KB_MAX_LINEAR_CORRECTION, 0.0f);
  moved = false;
  if (skipZero && C == 0.0f) return ok;   // the impulse is -0 / K and moves nothing
  const V2 rA = point - cA;
  const V2 rB = point - cB;
  const float rnA = cross(rA, normal);
  const float rnB = cross(rB, normal);
  const float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
  float impulse;
  if (EXACT_OPS) {
    impulse = K > 0.0f ? -C / K : 0.0f;
  } else {
    bad |= !(KB_DIV_WINDOW_POS(K) && -C >= 1.0842021724855044e-19f);   // (0 < -C <= 0.2; K <= 0: the exact pass answers)
    impulse = kb_div_raw(-C, K);
  }
  const V2 P = impulse * normal;
  cA = cA - mA * P;
  cB = cB + mB * P;
  a1 = make_float4(cA.x, cA.y, a0.z - iA * cross(rA, P), a0.w);
  b1 = make_float4(cB.x, cB.y, b0.z + iB * cross(rB, P), b0.w);
  moved = true;
  return ok;
}

// kb_position_pair_t's exact pass, out of line: called (in practice never) AFTER the straight-line results were stored, with the
// rows as they were before (by value: nothing of the hot path lives in local memory); it stores the exact rows itself --
// the old ones if the exact pass moves nothing.  wA / wB: shared-window addresses of the rows (0: do not store).
__device__ __noinline__ bool kb_position_pair_cold(uint32_t wA, uint32_t wB, float4 a0, float4 b0, float radiusA, float radiusB, float mA,
                                                float iA, float mB, float iB, float baumgarte, float limit, bool skipZero) {
  bool bad = false, moved;
  float4 a1, b1;
  const bool ok = kb_position_pair_t<true>(a0, b0, radiusA, radiusB, mA, iA, mB, iB, baumgarte, limit, skipZero, a1, b1, moved, bad);
  if (wA != 0u) sts_f4(wA, moved ? a1 : a0);
  if (wB != 0u) sts_f4(wB, moved ? b1 : b0);
  return ok;
}

// ---- per-body steps of b2Island::Solve / SolveTOI
// b2Island::Solve's velocity damping factor over h for a damping coefficient c: mode 0 is 1 / (1 + h c) (Box2D >= 2.3.1),
// mode 1 clamp(1 - h c, 0, 1)
__device__ __forceinline__ float kb_damping(int mode, float h, float c) {
  return mode == 0 ? 1.0f / (1.0f + h * c) : b2clamp(1.0f - h * c, 0.0f, 1.0f);
}

// position integration over h of p = (c.x, c.y, a, -) with v = (v.x, v.y, w, -), which the maximum translation and
// rotation per step clamp first
__device__ __forceinline__ void kb_integrate_position(float4& p, float4& v, float h) {
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
}

// b2Sweep::Advance(alpha) of sw = (c0.x, c0.y, a0, alpha0) towards the body's p = (c.x, c.y, a, -)
__device__ __forceinline__ void kb_sweep_advance(float4& sw, const float4& p, float alpha) {
  const float beta = (alpha - sw.w) / (1.0f - sw.w);
  sw.x += beta * (p.x - sw.x);
  sw.y += beta * (p.y - sw.y);
  sw.z += beta * (p.z - sw.z);
  sw.w = alpha;
}

// a body's sleep time after a step of h: back to zero while it moves faster than the sleep tolerances
__device__ __forceinline__ float kb_sleep_time(const float4& v, float sleepTime, float h) {
  const float linTolSqr = KB_LIN_SLEEP_TOL * KB_LIN_SLEEP_TOL;
  const float angTolSqr = KB_ANG_SLEEP_TOL * KB_ANG_SLEEP_TOL;
  if (v.z * v.z > angTolSqr || dot(mk(v.x, v.y), mk(v.x, v.y)) > linTolSqr) return 0.0f;
  return sleepTime + h;
}

}  // namespace kb
