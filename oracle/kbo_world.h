// CPU ORACLE -- TEST INFRASTRUCTURE ONLY (see kbo_math.h header).  PARITY UNPINNED.
//
// kbo_world.h -- object-per-world restatement of the Box2D 2.3.x subset gym_kilobots exercises
// through b2World.Step (envs/kilobots_env.py:187): bodies, circle/polygon/chain-edge fixtures,
// fat-AABB broadphase, persistent contacts with LIFO lists, island DFS, sequential-impulse
// contact solver, sleeping, and TOI against the static table.  Deliberately naive and pointer
// based (Box2D's own data-structure orderings), nothing like the CUDA kernel's layout.
#pragma once
#include <cstdint>
#include <vector>

#include "kbo_math.h"

namespace kbo {

enum ShapeType { kCircle = 0, kEdge = 1, kPolygon = 2 };
enum ManifoldType { kManifoldCircles = 0, kManifoldFaceA = 1, kManifoldFaceB = 2 };
enum FeatureType { kFeatureVertex = 0, kFeatureFace = 1 };

struct ContactFeature {
  uint8_t indexA, indexB, typeA, typeB;
};
union ContactID {
  ContactFeature cf;
  uint32_t key;
};
struct ManifoldPoint {
  Vec2 localPoint;
  float normalImpulse = 0.0f;
  float tangentImpulse = 0.0f;
  ContactID id;
  ManifoldPoint() { id.key = 0; }
};
struct Manifold {
  ManifoldPoint points[kMaxManifoldPoints];
  Vec2 localNormal;
  Vec2 localPoint;
  int type = kManifoldCircles;
  int pointCount = 0;
};
struct ClipVertex {
  Vec2 v;
  ContactID id;
};

struct MassData {
  float mass;
  Vec2 center;
  float I;
};

// One collision shape.  kEdge is one child of the table's b2ChainShape (b2ChainShape::GetChildEdge).
struct Shape {
  int type = kCircle;
  float radius = 0.0f;
  // circle
  Vec2 p;
  // polygon
  int count = 0;
  Vec2 vertices[kMaxPolygonVertices];
  Vec2 normals[kMaxPolygonVertices];
  Vec2 centroid;
  // edge
  Vec2 v0, v1, v2, v3;
  bool hasVertex0 = false, hasVertex3 = false;

  void SetAsBox(float hx, float hy);
  void SetPolygon(const Vec2* verts, int n);
  void ComputeAABB(AABB* aabb, const Xf& xf) const;
  void ComputeMass(MassData* md, float density) const;
};

struct Body;
struct Contact;

struct Fixture {
  Shape shape;
  Body* body = nullptr;
  float density = 0.0f, friction = 0.2f, restitution = 0.0f;
  int proxyId = -1;  // == index into World::proxies; monotone in creation order (SURVEY B.7)
  AABB fatAABB;      // b2DynamicTree leaf AABB
};

struct ContactEdge {
  Body* other = nullptr;
  Contact* contact = nullptr;
  ContactEdge* prev = nullptr;
  ContactEdge* next = nullptr;
};

struct Contact {
  enum { kIslandFlag = 1, kTouchingFlag = 2, kEnabledFlag = 4, kToiFlag = 32 };
  uint32_t flags = kEnabledFlag;
  Contact* prev = nullptr;
  Contact* next = nullptr;
  ContactEdge nodeA, nodeB;
  Fixture* fixtureA = nullptr;
  Fixture* fixtureB = nullptr;
  Manifold manifold;
  int toiCount = 0;
  float toi = 1.0f;
  float friction = 0.0f, restitution = 0.0f;
  void Evaluate(Manifold* m, const Xf& xfA, const Xf& xfB) const;
  void Update();
  bool IsTouching() const { return (flags & kTouchingFlag) != 0; }
  bool IsEnabled() const { return (flags & kEnabledFlag) != 0; }
};

struct Body {
  enum { kIslandFlag = 1, kAwakeFlag = 2 };
  bool isStatic = false;
  uint32_t flags = kAwakeFlag;
  int islandIndex = 0;
  Xf xf;
  Sweep sweep;
  Vec2 linearVelocity;
  float angularVelocity = 0.0f;
  float mass = 0.0f, invMass = 0.0f, I = 0.0f, invI = 0.0f;
  float linearDamping = 0.0f, angularDamping = 0.0f;
  float sleepTime = 0.0f;
  std::vector<Fixture*> fixtures;  // creation order; Box2D's m_fixtureList is this reversed
  ContactEdge* contactList = nullptr;
  int index = -1;  // creation index among dynamic bodies

  bool IsAwake() const { return (flags & kAwakeFlag) != 0; }
  void SetAwake(bool flag);
  void SetLinearVelocity(const Vec2& v);
  void SetAngularVelocity(float w);
  void SynchronizeTransform();
  void Advance(float alpha);
  void ResetMassData();
  Vec2 GetWorldPoint(const Vec2& lp) const { return Mul(xf, lp); }
  Vec2 GetWorldVector(const Vec2& lv) const { return Mul(xf.q, lv); }
};

struct WorldCounters {
  uint64_t substeps = 0, contacts = 0, points = 0, levels = 0, posIters = 0, toiEvents = 0,
           pairTests = 0, islands = 0;
};

struct World {
  // switches (SURVEY B.9)
  int dampingMode = 0;
  bool continuousPhysics = true;
  bool allowSleep = true;

  Body* table = nullptr;
  std::vector<Body*> bodies;       // dynamic bodies in creation order; Box2D's m_bodyList is reversed
  std::vector<Fixture*> proxies;   // all proxies in creation (= proxy id) order
  std::vector<int> moveBuffer;
  Contact* contactList = nullptr;
  int contactCount = 0;
  bool newFixture = false;
  WorldCounters counters;

  World() = default;
  ~World();
  World(const World&) = delete;
  World& operator=(const World&) = delete;

  void CreateTable(float x0, float y0, float x1, float y1, int edges, float friction);
  Body* CreateBody(float px, float py, float angle, float linearDamping, float angularDamping);
  Fixture* CreateFixture(Body* b, const Shape& shape, float density, float friction, float restitution);
  void SetTransform(Body* b, float px, float py, float angle);
  void Step(float dt, int velocityIterations, int positionIterations);

  // b2ContactManager
  void FindNewContacts();
  void AddPair(Fixture* fA, Fixture* fB);
  void Collide();
  void DestroyContact(Contact* c);
  // b2World
  void Solve(float dt, int velocityIterations, int positionIterations);
  void SolveTOI(float dt, int velocityIterations);
  void SynchronizeFixtures(Body* b);
  void MoveProxy(Fixture* f, const AABB& aabb, const Vec2& displacement);
};

// narrowphase (kbo_collide.cpp)
void CollideCircles(Manifold* m, const Shape* circleA, const Xf& xfA, const Shape* circleB, const Xf& xfB);
void CollidePolygonAndCircle(Manifold* m, const Shape* polyA, const Xf& xfA, const Shape* circleB, const Xf& xfB);
void CollidePolygons(Manifold* m, const Shape* polyA, const Xf& xfA, const Shape* polyB, const Xf& xfB);
void CollideEdgeAndCircle(Manifold* m, const Shape* edgeA, const Xf& xfA, const Shape* circleB, const Xf& xfB);
void CollideEdgeAndPolygon(Manifold* m, const Shape* edgeA, const Xf& xfA, const Shape* polyB, const Xf& xfB);

// continuous collision (kbo_toi.cpp)
struct TOIInput {
  const Shape* shapeA;
  const Shape* shapeB;
  Sweep sweepA, sweepB;
  float tMax;
};
struct TOIOutput {
  enum State { kUnknown, kFailed, kOverlapped, kTouching, kSeparated };
  State state;
  float t;
};
void TimeOfImpact(TOIOutput* out, const TOIInput* in);
// b2Distance (useRadii = false) of the core shapes with a fresh simplex cache; *simplexCount = the cache's count
float DistanceCore(const Shape* shapeA, const Xf& xfA, const Shape* shapeB, const Xf& xfB, int* simplexCount);

// child i of the table chain (kbo_world.cpp)
Shape MakeChainEdge(float x0, float y0, float x1, float y1, int edges, int i);

// contact solver over an island (kbo_solver.cpp)
struct Position { Vec2 c; float a; };
struct Velocity { Vec2 v; float w; };
struct VelocityConstraintPoint {
  Vec2 rA, rB;
  float normalImpulse, tangentImpulse, normalMass, tangentMass, velocityBias;
};
struct ContactVelocityConstraint {
  VelocityConstraintPoint points[kMaxManifoldPoints];
  Vec2 normal;
  Mat22 normalMass, K;
  int indexA, indexB;
  float invMassA, invMassB, invIA, invIB;
  float friction, restitution;
  int pointCount;
  int contactIndex;
};
struct ContactPositionConstraint {
  Vec2 localPoints[kMaxManifoldPoints];
  Vec2 localNormal, localPoint;
  int indexA, indexB;
  float invMassA, invMassB;
  Vec2 localCenterA, localCenterB;
  float invIA, invIB;
  int type;
  float radiusA, radiusB;
  int pointCount;
};
struct ContactSolver {
  ContactSolver(const std::vector<Contact*>& contacts, std::vector<Position>* positions,
                std::vector<Velocity>* velocities, float dtRatio, bool warmStarting);
  void InitializeVelocityConstraints();
  void WarmStart();
  void SolveVelocityConstraints();
  void StoreImpulses();
  bool SolvePositionConstraints();
  bool SolveTOIPositionConstraints(int toiIndexA, int toiIndexB);

  const std::vector<Contact*>& contacts;
  std::vector<Position>& positions;
  std::vector<Velocity>& velocities;
  std::vector<ContactVelocityConstraint> vcs;
  std::vector<ContactPositionConstraint> pcs;
};

}  // namespace kbo
