// CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED (see kbo_math.h).
// Restates b2World::Step / Solve / SolveTOI, b2ContactManager, b2BroadPhase (fat AABBs + move
// buffer + sorted pair buffer; the dynamic tree itself is replaced by an all-proxies scan, which
// yields the same pair set -- SURVEY.md B.6), b2Island::Solve / SolveTOI, b2Body and b2Contact of
// Box2D 2.3.x, as driven by gym_kilobots/envs/kilobots_env.py:45-51,187-188,217-219 and
// lib/body.py:32-38.
#include "kbo_world.h"

#include <algorithm>
#include <cmath>

namespace kbo {

// ------------------------------------------------------------------------------------- b2Body
void Body::SetAwake(bool flag) {
  if (flag) {
    if ((flags & kAwakeFlag) == 0) {
      flags |= kAwakeFlag;
      sleepTime = 0.0f;
    }
  } else {
    flags &= ~kAwakeFlag;
    sleepTime = 0.0f;
    linearVelocity.SetZero();
    angularVelocity = 0.0f;
  }
}

void Body::SetLinearVelocity(const Vec2& v) {
  if (isStatic) return;
  if (Dot(v, v) > 0.0f) SetAwake(true);
  linearVelocity = v;
}

void Body::SetAngularVelocity(float w) {
  if (isStatic) return;
  if (w * w > 0.0f) SetAwake(true);
  angularVelocity = w;
}

void Body::SynchronizeTransform() {
  xf.q.Set(sweep.a);
  xf.p = sweep.c - Mul(xf.q, sweep.localCenter);
}

void Body::Advance(float alpha) {
  sweep.Advance(alpha);
  sweep.c = sweep.c0;
  sweep.a = sweep.a0;
  xf.q.Set(sweep.a);
  xf.p = sweep.c - Mul(xf.q, sweep.localCenter);
}

void Body::ResetMassData() {
  mass = 0.0f;
  invMass = 0.0f;
  I = 0.0f;
  invI = 0.0f;
  sweep.localCenter.SetZero();
  if (isStatic) {
    sweep.c0 = xf.p;
    sweep.c = xf.p;
    sweep.a0 = sweep.a;
    return;
  }
  Vec2 localCenter(0.0f, 0.0f);
  // Box2D walks m_fixtureList, which is LIFO: last created fixture first.
  for (int k = (int)fixtures.size() - 1; k >= 0; --k) {
    Fixture* f = fixtures[k];
    if (f->density == 0.0f) continue;
    MassData md;
    f->shape.ComputeMass(&md, f->density);
    mass += md.mass;
    localCenter += md.mass * md.center;
    I += md.I;
  }
  if (mass > 0.0f) {
    invMass = 1.0f / mass;
    localCenter *= invMass;
  } else {
    mass = 1.0f;
    invMass = 1.0f;
  }
  if (I > 0.0f) {
    I -= mass * Dot(localCenter, localCenter);
    invI = 1.0f / I;
  } else {
    I = 0.0f;
    invI = 0.0f;
  }
  Vec2 oldCenter = sweep.c;
  sweep.localCenter = localCenter;
  sweep.c0 = sweep.c = Mul(xf, sweep.localCenter);
  linearVelocity += Cross(angularVelocity, sweep.c - oldCenter);
}

// ---------------------------------------------------------------------------------- b2Contact
void Contact::Evaluate(Manifold* m, const Xf& xfA, const Xf& xfB) const {
  const Shape* sA = &fixtureA->shape;
  const Shape* sB = &fixtureB->shape;
  if (sA->type == kCircle && sB->type == kCircle) CollideCircles(m, sA, xfA, sB, xfB);
  else if (sA->type == kPolygon && sB->type == kCircle) CollidePolygonAndCircle(m, sA, xfA, sB, xfB);
  else if (sA->type == kPolygon && sB->type == kPolygon) CollidePolygons(m, sA, xfA, sB, xfB);
  else if (sA->type == kEdge && sB->type == kCircle) CollideEdgeAndCircle(m, sA, xfA, sB, xfB);
  else if (sA->type == kEdge && sB->type == kPolygon) CollideEdgeAndPolygon(m, sA, xfA, sB, xfB);
  else m->pointCount = 0;
}

void Contact::Update() {
  Manifold oldManifold = manifold;
  flags |= kEnabledFlag;
  bool touching = false;
  bool wasTouching = (flags & kTouchingFlag) == kTouchingFlag;
  Body* bodyA = fixtureA->body;
  Body* bodyB = fixtureB->body;
  Evaluate(&manifold, bodyA->xf, bodyB->xf);
  touching = manifold.pointCount > 0;
  for (int i = 0; i < manifold.pointCount; ++i) {
    ManifoldPoint* mp2 = manifold.points + i;
    mp2->normalImpulse = 0.0f;
    mp2->tangentImpulse = 0.0f;
    ContactID id2 = mp2->id;
    for (int j = 0; j < oldManifold.pointCount; ++j) {
      ManifoldPoint* mp1 = oldManifold.points + j;
      if (mp1->id.key == id2.key) {
        mp2->normalImpulse = mp1->normalImpulse;
        mp2->tangentImpulse = mp1->tangentImpulse;
        break;
      }
    }
  }
  if (touching != wasTouching) {
    bodyA->SetAwake(true);
    bodyB->SetAwake(true);
  }
  if (touching) flags |= kTouchingFlag;
  else flags &= ~kTouchingFlag;
}

// ------------------------------------------------------------------------------------ b2World
World::~World() {
  Contact* c = contactList;
  while (c) {
    Contact* n = c->next;
    delete c;
    c = n;
  }
  for (Fixture* f : proxies) delete f;
  for (Body* b : bodies) delete b;
  delete table;
}

// Child i of the table's chain shape, kilobots_env.py:46-51 (b2ChainShape::GetChildEdge).  edges == 3: open chain
// (b2ChainShape::CreateChain, no ghost vertices at the ends); edges == 4: closed loop (CreateLoop).
Shape MakeChainEdge(float x0, float y0, float x1, float y1, int edges, int i) {
  Vec2 v[5] = {Vec2(x0, y1), Vec2(x0, y0), Vec2(x1, y0), Vec2(x1, y1), Vec2(x0, y1)};
  const int count = edges == 4 ? 5 : 4;  // b2ChainShape::m_count
  const bool loop = edges == 4;
  Shape s;
  s.type = kEdge;
  s.radius = kPolygonRadius;
  s.v1 = v[i];
  s.v2 = v[i + 1];
  if (i > 0) {
    s.v0 = v[i - 1];
    s.hasVertex0 = true;
  } else {
    s.v0 = loop ? v[count - 2] : Vec2(0.0f, 0.0f);
    s.hasVertex0 = loop;
  }
  if (i < count - 2) {
    s.v3 = v[i + 2];
    s.hasVertex3 = true;
  } else {
    s.v3 = loop ? v[1] : Vec2(0.0f, 0.0f);
    s.hasVertex3 = loop;
  }
  return s;
}

// Static table + chain shape.  One proxy per chain child, created first so the table's proxy ids are the lowest.
void World::CreateTable(float x0, float y0, float x1, float y1, int edges, float friction) {
  table = new Body();
  table->isStatic = true;
  table->xf.p.SetZero();
  table->xf.q.Set(0.0f);
  table->index = -1;
  if (edges <= 0) return;
  for (int i = 0; i < edges; ++i) {
    Shape s = MakeChainEdge(x0, y0, x1, y1, edges, i);
    Fixture* f = new Fixture();
    f->shape = s;
    f->body = table;
    f->density = 0.0f;
    f->friction = friction;
    f->restitution = 0.0f;
    AABB aabb;
    s.ComputeAABB(&aabb, table->xf);
    Vec2 r(kAabbExtension, kAabbExtension);
    f->fatAABB.lowerBound = aabb.lowerBound - r;
    f->fatAABB.upperBound = aabb.upperBound + r;
    f->proxyId = (int)proxies.size();
    proxies.push_back(f);
    moveBuffer.push_back(f->proxyId);
    table->fixtures.push_back(f);
  }
  newFixture = true;
}

// b2World::CreateBody with the b2BodyDef the reference fills in lib/body.py:32-36, followed by
// the explicit zero velocities of :37-38.
Body* World::CreateBody(float px, float py, float angle, float linearDamping, float angularDamping) {
  Body* b = new Body();
  b->xf.p.Set(px, py);
  b->xf.q.Set(angle);
  b->sweep.localCenter.SetZero();
  b->sweep.c0 = b->xf.p;
  b->sweep.c = b->xf.p;
  b->sweep.a0 = angle;
  b->sweep.a = angle;
  b->sweep.alpha0 = 0.0f;
  b->linearDamping = linearDamping;
  b->angularDamping = angularDamping;
  b->mass = 1.0f;
  b->invMass = 1.0f;
  b->index = (int)bodies.size();
  bodies.push_back(b);
  return b;
}

// b2Body::CreateFixture -> b2Fixture::CreateProxies -> b2BroadPhase::CreateProxy (fat AABB =
// aabb +- aabbExtension, proxy buffered as moved) -> ResetMassData.
Fixture* World::CreateFixture(Body* b, const Shape& shape, float density, float friction,
                              float restitution) {
  Fixture* f = new Fixture();
  f->shape = shape;
  f->body = b;
  f->density = density;
  f->friction = friction;
  f->restitution = restitution;
  AABB aabb;
  f->shape.ComputeAABB(&aabb, b->xf);
  Vec2 r(kAabbExtension, kAabbExtension);
  f->fatAABB.lowerBound = aabb.lowerBound - r;
  f->fatAABB.upperBound = aabb.upperBound + r;
  f->proxyId = (int)proxies.size();
  proxies.push_back(f);
  moveBuffer.push_back(f->proxyId);
  b->fixtures.push_back(f);
  if (density > 0.0f) b->ResetMassData();
  newFixture = true;
  return f;
}

// b2Body::SetTransform (pybox2d: body.position = ..., body.angle = ...; lib/body.py:54-69).
void World::SetTransform(Body* b, float px, float py, float angle) {
  b->xf.q.Set(angle);
  b->xf.p.Set(px, py);
  b->sweep.c = Mul(b->xf, b->sweep.localCenter);
  b->sweep.a = angle;
  b->sweep.c0 = b->sweep.c;
  b->sweep.a0 = angle;
  for (int k = (int)b->fixtures.size() - 1; k >= 0; --k) {
    Fixture* f = b->fixtures[k];
    AABB aabb1, aabb2, aabb;
    f->shape.ComputeAABB(&aabb1, b->xf);
    f->shape.ComputeAABB(&aabb2, b->xf);
    aabb.Combine(aabb1, aabb2);
    MoveProxy(f, aabb, Vec2(0.0f, 0.0f));
  }
}

void World::MoveProxy(Fixture* f, const AABB& aabb, const Vec2& displacement) {
  if (f->fatAABB.Contains(aabb)) return;
  AABB b = aabb;
  Vec2 r(kAabbExtension, kAabbExtension);
  b.lowerBound = b.lowerBound - r;
  b.upperBound = b.upperBound + r;
  Vec2 d = kAabbMultiplier * displacement;
  if (d.x < 0.0f) b.lowerBound.x += d.x;
  else b.upperBound.x += d.x;
  if (d.y < 0.0f) b.lowerBound.y += d.y;
  else b.upperBound.y += d.y;
  f->fatAABB = b;
  moveBuffer.push_back(f->proxyId);
}

void World::SynchronizeFixtures(Body* b) {
  Xf xf1;
  xf1.q.Set(b->sweep.a0);
  xf1.p = b->sweep.c0 - Mul(xf1.q, b->sweep.localCenter);
  for (int k = (int)b->fixtures.size() - 1; k >= 0; --k) {
    Fixture* f = b->fixtures[k];
    AABB aabb1, aabb2, aabb;
    f->shape.ComputeAABB(&aabb1, xf1);
    f->shape.ComputeAABB(&aabb2, b->xf);
    aabb.Combine(aabb1, aabb2);
    Vec2 displacement = b->xf.p - xf1.p;
    MoveProxy(f, aabb, displacement);
  }
}

// b2BroadPhase::UpdatePairs + b2ContactManager::AddPair
void World::FindNewContacts() {
  std::vector<std::pair<int, int>> pairBuffer;
  for (int queryId : moveBuffer) {
    const AABB& fat = proxies[queryId]->fatAABB;
    for (int id = 0; id < (int)proxies.size(); ++id) {
      if (id == queryId) continue;
      ++counters.pairTests;
      if (!TestOverlap(proxies[id]->fatAABB, fat)) continue;
      pairBuffer.emplace_back(std::min(id, queryId), std::max(id, queryId));
    }
  }
  moveBuffer.clear();
  std::sort(pairBuffer.begin(), pairBuffer.end());
  size_t i = 0;
  while (i < pairBuffer.size()) {
    std::pair<int, int> primary = pairBuffer[i];
    AddPair(proxies[primary.first], proxies[primary.second]);
    ++i;
    while (i < pairBuffer.size() && pairBuffer[i] == primary) ++i;
  }
}

void World::AddPair(Fixture* fixtureA, Fixture* fixtureB) {
  Body* bodyA = fixtureA->body;
  Body* bodyB = fixtureB->body;
  if (bodyA == bodyB) return;
  for (ContactEdge* edge = bodyB->contactList; edge; edge = edge->next) {
    if (edge->other == bodyA) {
      Fixture* fA = edge->contact->fixtureA;
      Fixture* fB = edge->contact->fixtureB;
      if (fA == fixtureA && fB == fixtureB) return;
      if (fA == fixtureB && fB == fixtureA) return;
    }
  }
  // b2Body::ShouldCollide: at least one body must be dynamic.
  if (bodyA->isStatic && bodyB->isStatic) return;
  // b2Contact::Create: the type register may swap the fixtures (chain < polygon < circle as A).
  auto rank = [](const Fixture* f) { return f->shape.type == kEdge ? 0 : (f->shape.type == kPolygon ? 1 : 2); };
  if (rank(fixtureA) > rank(fixtureB)) std::swap(fixtureA, fixtureB);
  bodyA = fixtureA->body;
  bodyB = fixtureB->body;
  Contact* c = new Contact();
  c->fixtureA = fixtureA;
  c->fixtureB = fixtureB;
  c->friction = sqrtf(fixtureA->friction * fixtureB->friction);
  c->restitution = fixtureA->restitution > fixtureB->restitution ? fixtureA->restitution : fixtureB->restitution;
  c->prev = nullptr;
  c->next = contactList;
  if (contactList) contactList->prev = c;
  contactList = c;
  c->nodeA.contact = c;
  c->nodeA.other = bodyB;
  c->nodeA.prev = nullptr;
  c->nodeA.next = bodyA->contactList;
  if (bodyA->contactList) bodyA->contactList->prev = &c->nodeA;
  bodyA->contactList = &c->nodeA;
  c->nodeB.contact = c;
  c->nodeB.other = bodyA;
  c->nodeB.prev = nullptr;
  c->nodeB.next = bodyB->contactList;
  if (bodyB->contactList) bodyB->contactList->prev = &c->nodeB;
  bodyB->contactList = &c->nodeB;
  bodyA->SetAwake(true);
  bodyB->SetAwake(true);
  ++contactCount;
}

void World::DestroyContact(Contact* c) {
  Body* bodyA = c->fixtureA->body;
  Body* bodyB = c->fixtureB->body;
  if (c->prev) c->prev->next = c->next;
  if (c->next) c->next->prev = c->prev;
  if (c == contactList) contactList = c->next;
  if (c->nodeA.prev) c->nodeA.prev->next = c->nodeA.next;
  if (c->nodeA.next) c->nodeA.next->prev = c->nodeA.prev;
  if (&c->nodeA == bodyA->contactList) bodyA->contactList = c->nodeA.next;
  if (c->nodeB.prev) c->nodeB.prev->next = c->nodeB.next;
  if (c->nodeB.next) c->nodeB.next->prev = c->nodeB.prev;
  if (&c->nodeB == bodyB->contactList) bodyB->contactList = c->nodeB.next;
  // b2Contact::Destroy
  if (c->manifold.pointCount > 0) {
    bodyA->SetAwake(true);
    bodyB->SetAwake(true);
  }
  delete c;
  --contactCount;
}

void World::Collide() {
  Contact* c = contactList;
  while (c) {
    Fixture* fixtureA = c->fixtureA;
    Fixture* fixtureB = c->fixtureB;
    Body* bodyA = fixtureA->body;
    Body* bodyB = fixtureB->body;
    bool activeA = bodyA->IsAwake() && !bodyA->isStatic;
    bool activeB = bodyB->IsAwake() && !bodyB->isStatic;
    if (!activeA && !activeB) {
      c = c->next;
      continue;
    }
    bool overlap = TestOverlap(fixtureA->fatAABB, fixtureB->fatAABB);
    if (!overlap) {
      Contact* cNuke = c;
      c = cNuke->next;
      DestroyContact(cNuke);
      continue;
    }
    c->Update();
    c = c->next;
  }
}

void World::Step(float dt, int velocityIterations, int positionIterations) {
  if (newFixture) {
    FindNewContacts();
    newFixture = false;
  }
  ++counters.substeps;
  counters.contacts += (uint64_t)contactCount;
  Collide();
  if (dt > 0.0f) Solve(dt, velocityIterations, positionIterations);
  if (continuousPhysics && dt > 0.0f) SolveTOI(dt, velocityIterations);
}

// b2World::Solve: island DFS over LIFO body / contact-edge lists, then b2Island::Solve.
void World::Solve(float dt, int velocityIterations, int positionIterations) {
  for (Body* b : bodies) b->flags &= ~Body::kIslandFlag;
  table->flags &= ~Body::kIslandFlag;
  for (Contact* c = contactList; c; c = c->next) c->flags &= ~Contact::kIslandFlag;

  std::vector<Body*> stack;
  std::vector<Body*> islandBodies;
  std::vector<Contact*> islandContacts;
  std::vector<Position> positions;
  std::vector<Velocity> velocities;
  const float h = dt;

  for (int si = (int)bodies.size() - 1; si >= 0; --si) {  // m_bodyList: newest body first
    Body* seed = bodies[si];
    if (seed->flags & Body::kIslandFlag) continue;
    if (!seed->IsAwake()) continue;
    islandBodies.clear();
    islandContacts.clear();
    stack.clear();
    stack.push_back(seed);
    seed->flags |= Body::kIslandFlag;
    while (!stack.empty()) {
      Body* b = stack.back();
      stack.pop_back();
      b->islandIndex = (int)islandBodies.size();
      islandBodies.push_back(b);
      b->SetAwake(true);
      if (b->isStatic) continue;
      for (ContactEdge* ce = b->contactList; ce; ce = ce->next) {
        Contact* contact = ce->contact;
        if (contact->flags & Contact::kIslandFlag) continue;
        if (!contact->IsEnabled() || !contact->IsTouching()) continue;
        islandContacts.push_back(contact);
        contact->flags |= Contact::kIslandFlag;
        Body* other = ce->other;
        if (other->flags & Body::kIslandFlag) continue;
        stack.push_back(other);
        other->flags |= Body::kIslandFlag;
      }
    }

    // ---- b2Island::Solve ----
    ++counters.islands;
    const int bodyCount = (int)islandBodies.size();
    positions.resize(bodyCount);
    velocities.resize(bodyCount);
    for (int i = 0; i < bodyCount; ++i) {
      Body* b = islandBodies[i];
      Vec2 c = b->sweep.c;
      float a = b->sweep.a;
      Vec2 v = b->linearVelocity;
      float w = b->angularVelocity;
      b->sweep.c0 = b->sweep.c;
      b->sweep.a0 = b->sweep.a;
      if (!b->isStatic) {
        // gravity = 0 and no forces are ever applied (kilobots_env.py:45,188): v += h*0.
        if (dampingMode == 0) {
          v *= 1.0f / (1.0f + h * b->linearDamping);
          w *= 1.0f / (1.0f + h * b->angularDamping);
        } else {
          v *= Clamp(1.0f - h * b->linearDamping, 0.0f, 1.0f);
          w *= Clamp(1.0f - h * b->angularDamping, 0.0f, 1.0f);
        }
      }
      positions[i].c = c;
      positions[i].a = a;
      velocities[i].v = v;
      velocities[i].w = w;
    }
    ContactSolver solver(islandContacts, &positions, &velocities, 1.0f, true);
    solver.InitializeVelocityConstraints();
    solver.WarmStart();
    for (int i = 0; i < velocityIterations; ++i) solver.SolveVelocityConstraints();
    solver.StoreImpulses();
    for (const Contact* ic : islandContacts) counters.points += (uint64_t)ic->manifold.pointCount;
    for (int i = 0; i < bodyCount; ++i) {
      Vec2 c = positions[i].c;
      float a = positions[i].a;
      Vec2 v = velocities[i].v;
      float w = velocities[i].w;
      Vec2 translation = h * v;
      if (Dot(translation, translation) > kMaxTranslationSquared) {
        float ratio = kMaxTranslation / translation.Length();
        v *= ratio;
      }
      float rotation = h * w;
      if (rotation * rotation > kMaxRotationSquared) {
        float ratio = kMaxRotation / Abs(rotation);
        w *= ratio;
      }
      c += h * v;
      a += h * w;
      positions[i].c = c;
      positions[i].a = a;
      velocities[i].v = v;
      velocities[i].w = w;
    }
    bool positionSolved = false;
    for (int i = 0; i < positionIterations; ++i) {
      ++counters.posIters;
      bool contactsOkay = solver.SolvePositionConstraints();
      if (contactsOkay) {
        positionSolved = true;
        break;
      }
    }
    for (int i = 0; i < bodyCount; ++i) {
      Body* body = islandBodies[i];
      body->sweep.c = positions[i].c;
      body->sweep.a = positions[i].a;
      body->linearVelocity = velocities[i].v;
      body->angularVelocity = velocities[i].w;
      body->SynchronizeTransform();
    }
    if (allowSleep) {
      float minSleepTime = kMaxFloat;
      const float linTolSqr = kLinearSleepTolerance * kLinearSleepTolerance;
      const float angTolSqr = kAngularSleepTolerance * kAngularSleepTolerance;
      for (int i = 0; i < bodyCount; ++i) {
        Body* b = islandBodies[i];
        if (b->isStatic) continue;
        if (b->angularVelocity * b->angularVelocity > angTolSqr ||
            Dot(b->linearVelocity, b->linearVelocity) > linTolSqr) {
          b->sleepTime = 0.0f;
          minSleepTime = 0.0f;
        } else {
          b->sleepTime += h;
          minSleepTime = Min(minSleepTime, b->sleepTime);
        }
      }
      if (minSleepTime >= kTimeToSleep && positionSolved) {
        for (int i = 0; i < bodyCount; ++i) islandBodies[i]->SetAwake(false);
      }
    }
    for (int i = 0; i < bodyCount; ++i) {
      Body* b = islandBodies[i];
      if (b->isStatic) b->flags &= ~Body::kIslandFlag;
    }
  }

  for (int i = (int)bodies.size() - 1; i >= 0; --i) {
    Body* b = bodies[i];
    if ((b->flags & Body::kIslandFlag) == 0) continue;
    SynchronizeFixtures(b);
  }
  FindNewContacts();
}

// b2World::SolveTOI + b2Island::SolveTOI.  No bullets exist, so only contacts with the static
// table are ever candidates.
void World::SolveTOI(float dt, int velocityIterations) {
  for (Body* b : bodies) {
    b->flags &= ~Body::kIslandFlag;
    b->sweep.alpha0 = 0.0f;
  }
  table->flags &= ~Body::kIslandFlag;
  table->sweep.alpha0 = 0.0f;
  for (Contact* c = contactList; c; c = c->next) {
    c->flags &= ~(Contact::kToiFlag | Contact::kIslandFlag);
    c->toiCount = 0;
    c->toi = 1.0f;
  }

  for (;;) {
    Contact* minContact = nullptr;
    float minAlpha = 1.0f;
    for (Contact* c = contactList; c; c = c->next) {
      if (!c->IsEnabled()) continue;
      if (c->toiCount > kMaxSubSteps) continue;
      float alpha = 1.0f;
      if (c->flags & Contact::kToiFlag) {
        alpha = c->toi;
      } else {
        Fixture* fA = c->fixtureA;
        Fixture* fB = c->fixtureB;
        Body* bA = fA->body;
        Body* bB = fB->body;
        bool activeA = bA->IsAwake() && !bA->isStatic;
        bool activeB = bB->IsAwake() && !bB->isStatic;
        if (!activeA && !activeB) continue;
        bool collideA = bA->isStatic;  // IsBullet() || type != dynamic
        bool collideB = bB->isStatic;
        if (!collideA && !collideB) continue;
        float alpha0 = bA->sweep.alpha0;
        if (bA->sweep.alpha0 < bB->sweep.alpha0) {
          alpha0 = bB->sweep.alpha0;
          bA->sweep.Advance(alpha0);
        } else if (bB->sweep.alpha0 < bA->sweep.alpha0) {
          alpha0 = bA->sweep.alpha0;
          bB->sweep.Advance(alpha0);
        }
        TOIInput input;
        input.shapeA = &fA->shape;
        input.shapeB = &fB->shape;
        input.sweepA = bA->sweep;
        input.sweepB = bB->sweep;
        input.tMax = 1.0f;
        TOIOutput output;
        TimeOfImpact(&output, &input);
        float beta = output.t;
        if (output.state == TOIOutput::kTouching) alpha = Min(alpha0 + (1.0f - alpha0) * beta, 1.0f);
        else alpha = 1.0f;
        c->toi = alpha;
        c->flags |= Contact::kToiFlag;
      }
      if (alpha < minAlpha) {
        minContact = c;
        minAlpha = alpha;
      }
    }
    if (minContact == nullptr || 1.0f - 10.0f * kEpsilon < minAlpha) break;

    ++counters.toiEvents;
    Fixture* fA = minContact->fixtureA;
    Fixture* fB = minContact->fixtureB;
    Body* bA = fA->body;
    Body* bB = fB->body;
    Sweep backup1 = bA->sweep;
    Sweep backup2 = bB->sweep;
    bA->Advance(minAlpha);
    bB->Advance(minAlpha);
    minContact->Update();
    minContact->flags &= ~Contact::kToiFlag;
    ++minContact->toiCount;
    if (!minContact->IsEnabled() || !minContact->IsTouching()) {
      minContact->flags &= ~Contact::kEnabledFlag;
      bA->sweep = backup1;
      bB->sweep = backup2;
      bA->SynchronizeTransform();
      bB->SynchronizeTransform();
      continue;
    }
    bA->SetAwake(true);
    bB->SetAwake(true);

    std::vector<Body*> islandBodies;
    std::vector<Contact*> islandContacts;
    auto addBody = [&](Body* b) {
      b->islandIndex = (int)islandBodies.size();
      islandBodies.push_back(b);
    };
    addBody(bA);
    addBody(bB);
    islandContacts.push_back(minContact);
    bA->flags |= Body::kIslandFlag;
    bB->flags |= Body::kIslandFlag;
    minContact->flags |= Contact::kIslandFlag;

    Body* pair[2] = {bA, bB};
    for (int i = 0; i < 2; ++i) {
      Body* body = pair[i];
      if (body->isStatic) continue;
      for (ContactEdge* ce = body->contactList; ce; ce = ce->next) {
        if ((int)islandBodies.size() == 2 * kMaxTOIContacts) break;
        if ((int)islandContacts.size() == kMaxTOIContacts) break;
        Contact* contact = ce->contact;
        if (contact->flags & Contact::kIslandFlag) continue;
        Body* other = ce->other;
        if (!other->isStatic) continue;  // only static / kinematic / bullet bodies are added
        Sweep backup = other->sweep;
        if ((other->flags & Body::kIslandFlag) == 0) other->Advance(minAlpha);
        contact->Update();
        if (!contact->IsEnabled()) {
          other->sweep = backup;
          other->SynchronizeTransform();
          continue;
        }
        if (!contact->IsTouching()) {
          other->sweep = backup;
          other->SynchronizeTransform();
          continue;
        }
        contact->flags |= Contact::kIslandFlag;
        islandContacts.push_back(contact);
        if (other->flags & Body::kIslandFlag) continue;
        other->flags |= Body::kIslandFlag;
        addBody(other);
      }
    }

    // ---- b2Island::SolveTOI ----
    const float subDt = (1.0f - minAlpha) * dt;
    const int toiIndexA = bA->islandIndex;
    const int toiIndexB = bB->islandIndex;
    const int bodyCount = (int)islandBodies.size();
    std::vector<Position> positions(bodyCount);
    std::vector<Velocity> velocities(bodyCount);
    for (int i = 0; i < bodyCount; ++i) {
      Body* b = islandBodies[i];
      positions[i].c = b->sweep.c;
      positions[i].a = b->sweep.a;
      velocities[i].v = b->linearVelocity;
      velocities[i].w = b->angularVelocity;
    }
    ContactSolver solver(islandContacts, &positions, &velocities, 1.0f, false);
    for (int i = 0; i < 20; ++i) {
      bool contactsOkay = solver.SolveTOIPositionConstraints(toiIndexA, toiIndexB);
      if (contactsOkay) break;
    }
    islandBodies[toiIndexA]->sweep.c0 = positions[toiIndexA].c;
    islandBodies[toiIndexA]->sweep.a0 = positions[toiIndexA].a;
    islandBodies[toiIndexB]->sweep.c0 = positions[toiIndexB].c;
    islandBodies[toiIndexB]->sweep.a0 = positions[toiIndexB].a;
    solver.InitializeVelocityConstraints();
    for (int i = 0; i < velocityIterations; ++i) solver.SolveVelocityConstraints();
    const float h = subDt;
    for (int i = 0; i < bodyCount; ++i) {
      Vec2 c = positions[i].c;
      float a = positions[i].a;
      Vec2 v = velocities[i].v;
      float w = velocities[i].w;
      Vec2 translation = h * v;
      if (Dot(translation, translation) > kMaxTranslationSquared) {
        float ratio = kMaxTranslation / translation.Length();
        v *= ratio;
      }
      float rotation = h * w;
      if (rotation * rotation > kMaxRotationSquared) {
        float ratio = kMaxRotation / Abs(rotation);
        w *= ratio;
      }
      c += h * v;
      a += h * w;
      positions[i].c = c;
      positions[i].a = a;
      velocities[i].v = v;
      velocities[i].w = w;
      Body* body = islandBodies[i];
      body->sweep.c = c;
      body->sweep.a = a;
      body->linearVelocity = v;
      body->angularVelocity = w;
      body->SynchronizeTransform();
    }

    for (int i = 0; i < bodyCount; ++i) {
      Body* body = islandBodies[i];
      body->flags &= ~Body::kIslandFlag;
      if (body->isStatic) continue;
      SynchronizeFixtures(body);
      for (ContactEdge* ce = body->contactList; ce; ce = ce->next)
        ce->contact->flags &= ~(Contact::kToiFlag | Contact::kIslandFlag);
    }
    FindNewContacts();
  }
}

}  // namespace kbo
