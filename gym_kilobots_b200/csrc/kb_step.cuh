// kb_step.cuh -- one lane group (4, 8, 16 or 32 lanes of a warp) per environment; the whole
// KilobotsEnv.step (gym_kilobots/envs/kilobots_env.py:161-215) for that environment runs inside one
// kernel launch with bodies, fat AABBs, the persistent contact words, the light and the solver's
// constraint records resident in shared memory across all sub-steps of the action.
//
// Phases per sub-step (reference call sites in brackets):
//   light_step      [lib/light.py:59-75, 300-316, 237-253; kilobots_env.py:171-172]
//   sense_control   [lib/kilobot.py:54-55,188-189; lib/light.py:176-189; lib/kilobot.py:86-127,191-203,253-258,294-300,318-333]
//   collide         [Box2D b2ContactManager::Collide + b2Contact::Update, via b2World.Step kilobots_env.py:187]
//   solve           [b2World::Solve: island DFS, b2Island::Solve, b2ContactSolver; sleeping; SynchronizeFixtures]
//   find_new        [b2BroadPhase::UpdatePairs + b2ContactManager::AddPair]
//   solve_toi       [b2World::SolveTOI, kb_toi.cuh]
// Ordering contract: the persistent contact array is kept in creation order, so Box2D's LIFO world
// list / per-body contact lists are "descending array index"; the island DFS, the constraint order
// and therefore every float32 result follow Box2D's sequential-impulse order exactly.  Within that
// order, constraints are executed row by row (a row = constraints of one dependency level whose
// dynamic bodies are disjoint and whose predecessors are done), which is bit-identical to the
// sequential sweep.
#pragma once
#include "kb_narrow.cuh"
#include "kb_sample.cuh"

namespace kb {

// task layer (extension, include/kb_b200.h "Task layer"): constants of the handle's KbTaskDef
struct TaskConst {
  int32_t mode, object, maxSteps, pad;
  double wPos, wAng, stepPenalty, bonus, posTol, angTol;
};
// per-env task words (float64): target x y theta, then the KB_EPISODE_STATS statistics
#define KB_TASK_WORDS (3 + KB_EPISODE_STATS + 2)   /* + the task error at the start of the current env-step */

struct KernelArgs {
  Layout L;
  SwarmLayout W;                // large-swarm tier (kb_swarm.cuh); W.enabled == 0 for the lane-group kernels
  float* blobs;                 // [E][blobWords]
  const int32_t* envScene;      // [E]
  const ProxyConst* proxies;    // [S][Pp]
  const BodyConst* bodies;      // [S][Bp]
  const SceneConst* scenes;     // [S]
  const LightConst* lights;     // [numLights]
  int32_t numEnvs;
  int32_t envOffset;             // first env of this launch (kb_step_host pipelines the batch in chunks)
  // step
  const double* action;
  int32_t actionMode;
  float* obsKilobots;
  float* obsObjects;
  double* obsLight;
  float* reward;
  uint8_t* done;
  int32_t* status;
  TaskConst task;
  double* taskState;            // [E][KB_TASK_WORDS]
  float* obsFlat;               // [E][2N + L + 4M] or null
#ifdef KB_PROFILE
  unsigned long long* prof;     // [E][KB_PROF_SLOTS] cycles per phase (debug builds only)
#endif
  // reset
  const uint8_t* mask;
  const double* pose;
  const double* lightInit;
  const double* kbVel;
  // reset with on-device scene sampling (kb_sample.cuh): the kernel draws pose / lightInit itself into the handle's
  // sample buffers (samplePose == pose, sampleLight == lightInit), may switch the env's scene, and counts episodes
  const SamplerConst* sampler;
  double* samplePose;
  double* sampleLight;
  int32_t* envSceneW;
  uint32_t* episode;
  // several configurations (kb_set_sampler_mix): sampler[numConfigs]; a sampled reset draws the configuration from
  // configCdf [numConfigs] (cumulative weights, last entry 1) or, when that is null, takes sceneConfig[env's scene].
  // Appended so that the offsets of the step kernels' parameters stay where they were.
  const int32_t* sceneConfig;   // [S], -1 = no configuration
  const double* configCdf;
  int32_t numConfigs;
};

}  // namespace kb
#include "kb_env.cuh"   // lights, controllers and task layer of both tiers: they take KernelArgs
namespace kb {

// general-constraint record words (GR_WORDS per record, HBM/L2)
#define PF_IDX 0   /* bA | bB<<8 | vcPointCount<<16 | type<<24 | pointCount<<28 */
#define PF_AUX 1   /* contact index | island<<16 */
#define PF_NX 2
#define PF_NY 3
#define PF_RAX 4
#define PF_RAY 5
#define PF_RBX 6
#define PF_RBY 7
#define PF_NMASS 8
#define PF_NIMP 9

// touching-list word tl[t]: contact index | bA << 16 | bB << 22 | general << 28
#define TL_GEN (1u << 28)
// schedule item ent[e]: bA | bB << 6 | island << 12 | general << 18 | fast << 19 | row << 22 (10 bits)
#define IT_BA(x) ((int)((x) & 63u))
#define IT_BB(x) ((int)(((x) >> 6) & 63u))
#define IT_ISL(x) ((int)(((x) >> 12) & 63u))
#define IT_GEN (1u << 18)
#define IT_FAST (1u << 19)   /* set by storeSimple: circle manifold between two bodies whose transforms need no rotation */
#define IT_ROW(x) ((int)((x) >> 22))
#define IT_NONE 0xFFFFFFFFu

// All shared-memory accesses index this symbol so that the compiler emits LDS/STS with 32-bit
// addresses (a pointer kept in a struct decays to generic LD/ST).
extern __shared__ __align__(16) uint32_t kb_smem[];

// phase timers (only with -DKB_PROFILE; compiled out of the product library)
#define KB_PROF_SLOTS 16
#ifdef KB_PROFILE
#define KB_T(i)                          \
  do {                                   \
    if (UNI) __syncthreads();            \
    const long long now_ = clock64();    \
    tp[i] += now_ - tlast;               \
    tlast = now_;                        \
  } while (0)
#else
// block-wide rendezvous at the phase boundaries of uniform mode (step kernel only; every thread of the block is
// alive and the boundaries sit in block-uniform control flow): the warps of a block then walk the same code at
// the same time and share instruction-cache lines -- the instruction footprint of one sub-step is several times
// the L1.5 instruction cache, and without this the fetch stalls were ~20 % of all warp stalls (profiles/).
#ifndef KB_SYNC_PHASES
#define KB_SYNC_PHASES 0xFFFu   /* bit i: rendezvous at phase boundary i */
#endif
#define KB_T(i) do { if (UNI && ((KB_SYNC_PHASES >> (i)) & 1u)) __syncthreads(); } while (0)
#endif

// The layout a Sim reads its offsets, counts and constants from: the runtime Layout in the kernel parameters (held by
// reference), or a compile-time layout -- an empty struct whose members are static constexpr copies of one batch's
// Layout, generated by kb_create for the step kernel it compiles at run time (kb_jit.h).  Code reads s.L.x either way.
template <class LT>
struct LayoutHold {
  typedef LT type;
};
template <>
struct LayoutHold<Layout> {
  typedef const Layout& type;
};

template <int LPE, bool UNI, class LT = Layout>
struct Sim;
// out-of-line (cold) paths: the Sim travels BY VALUE so that the caller's copy stays in registers
template <int LPE, bool UNI, class LT> __device__ __noinline__ void warmStartGeneralNI(Sim<LPE, UNI, LT> s, int q);
template <int LPE, bool UNI, class LT> __device__ __noinline__ void solveVelocityGeneralNI(Sim<LPE, UNI, LT> s, int q);
template <int LPE, bool UNI, class LT> __device__ __noinline__ bool solvePositionGeneralNI(Sim<LPE, UNI, LT> s, int q);
template <int LPE, bool UNI, class LT> __device__ __noinline__ void initGeneralNI(Sim<LPE, UNI, LT> s, int q, int ci, uint32_t item);
template <int LPE, bool UNI, class LT> __device__ __noinline__ void storeGeneralNI(Sim<LPE, UNI, LT> s, int q);
template <int LPE, bool UNI, class LT> __device__ __noinline__ uint32_t solveTOINI(Sim<LPE, UNI, LT> s);

template <int LPE, bool UNI, class LT>
struct Sim {
  Group<LPE, UNI> g;
  typename LayoutHold<LT>::type L;
  uint32_t sa;                  // shared-window byte address of this env's shared-memory region
  float* blob;                  // this env's state blob in HBM
  const ProxyConst* px;         // scene proxies
  const BodyConst* bc;          // scene bodies
  const LightConst* lights;
  int S;                        // index of the static table in the body arrays (== L.B)
  // per-launch counter increments (lane 0's copy is flushed to the blob at the end)
  uint32_t nSub, nCon, nPts, nLvl, nPit, nToi, nTests, nIsl;
  float* genBase;               // where the general-constraint records of the current solve live
#ifdef KB_PROFILE
  long long tp[KB_PROF_SLOTS], tlast;
  unsigned long long* profOut;   // this env's row of the profile buffer (TOI internals add to slots 13..15 directly)
#endif

  __device__ __forceinline__ Sim(const LT& l) : L(l) {
    nSub = nCon = nPts = nLvl = nPit = nToi = nTests = nIsl = 0u;
    genBase = nullptr;
#ifdef KB_PROFILE
    for (int i = 0; i < KB_PROF_SLOTS; ++i) tp[i] = 0;
    tlast = clock64();
#endif
  }
  __device__ __forceinline__ void bind(int slot) {
    const uint32_t a0 = (uint32_t)__cvta_generic_to_shared(kb_smem) + (uint32_t)slot * (uint32_t)L.smemWords * 4u;
    // opaque move: keeps the base in a register instead of re-deriving it (CTA-rank read) at every use
    asm volatile("mov.u32 %0, %1;" : "=r"(sa) : "r"(a0));
  }

  // ---- typed views into shared memory (proxies standing in for references; see kb_types.cuh)
  __device__ __forceinline__ uint32_t wa(int w) const { return sa + 4u * (uint32_t)w; }  // byte address of word w
  __device__ __forceinline__ SU32 word(int w) const { return SU32{wa(w)}; }
  __device__ __forceinline__ SF4 pos4(int b) const { return SF4{wa(L.oPos + 4 * b)}; }     // cx cy a sleepTime
  __device__ __forceinline__ SF4 vel4(int b) const { return SF4{wa(L.oVel + 4 * b)}; }     // vx vy w flags
  __device__ __forceinline__ SF4 xf4(int b) const { return SF4{wa(L.oXf + 4 * b)}; }       // px py qs qc
  // the position the task and the observations read: xf.p
  __device__ __forceinline__ float2 obsPos(int b) const {
    const float4 x = xf4(b);
    return make_float2(x.x, x.y);
  }
  __device__ __forceinline__ SF4 fat4(int p) const { return SF4{wa(L.oFat + 4 * p)}; }     // lx ly ux uy
  __device__ __forceinline__ SF4 sweep4(int b) const { return SF4{wa(L.sSweep + 4 * b)}; } // c0x c0y a0 alpha0
  __device__ __forceinline__ SF2 oldq(int b) const { return SF2{wa(L.sOldQ + 2 * b)}; }    // xf.q at step start
  __device__ __forceinline__ SF4 bc4(int b) const { return SF4{wa(L.sBc + 4 * b)}; }       // invMass invI lcx lcy
  __device__ __forceinline__ SF4 rec4(int i) const { return SF4{wa(L.sRec + 4 * i)}; }     // 2 per schedule entry
  __device__ __forceinline__ SU32 cw(int i) const { return SU32{wa(L.oCw + i)}; }
  __device__ __forceinline__ SU32 hdr(int i) const { return SU32{wa(L.oHdr + i)}; }
  __device__ __forceinline__ SI32 isl(int b) const { return SI32{wa(L.sIsl + b)}; }
  __device__ __forceinline__ SU32 islflag(int i) const { return SU32{wa(L.sIslFlag + i)}; }
  __device__ __forceinline__ SU32 misc(int i) const { return SU32{wa(L.sMisc + i)}; }
  __device__ __forceinline__ SU32 adj(int p, int hi) const { return SU32{wa(L.sAdj + 2 * p + hi)}; }
  __device__ __forceinline__ SU32 bmask(int b, int w) const { return SU32{wa(L.sBmask + b * L.KW + w)}; }
  __device__ __forceinline__ SU32 tl(int t) const { return SU32{wa(L.sTl + t)}; }
  __device__ __forceinline__ SU32 ord(int p) const { return SU32{wa(L.sOrd + p)}; }
  __device__ __forceinline__ SU32 ent(int e) const { return SU32{wa(L.sEnt + e)}; }
  __device__ __forceinline__ SU16 entC(int e) const { return SU16{wa(L.sEntC) + 2u * (uint32_t)e}; }
  __device__ __forceinline__ SU32 lvlTab(int l) const { return SU32{wa(L.sLvlTab + l)}; }
  __device__ __forceinline__ SU32 lastLvl(int b) const { return SU32{wa(L.sLastLvl + b)}; }
  __device__ __forceinline__ SI32 stk(int i) const { return SI32{wa(L.sStack + i)}; }      // DFS stack / wakeAt
  __device__ __forceinline__ int pbody(int p) const { return (int)lds_u8(wa(L.sPb) + (uint32_t)p); }
  // proxy flags: bits 0-1 shape type, bit 2 friction == 0, bit 3 restitution == 0
  __device__ __forceinline__ int pflags(int p) const { return (int)lds_u8(wa(L.sPt) + (uint32_t)p); }
  __device__ __forceinline__ int ptype(int p) const { return pflags(p) & 3; }
  __device__ __forceinline__ int bkind(int b) const { return (int)lds_u8(wa(L.sBk) + (uint32_t)b); }
  __device__ __forceinline__ SF2 damp(int b) const { return SF2{wa(L.sDamp + 2 * b)}; }  // velocity damping factors
  __device__ __forceinline__ LCs lightConst(int l) const { return LCs{wa(L.sLc + LC_WORDS * l)}; }
  __device__ __forceinline__ float pradius(int p) const { return lds_f32(wa(L.sPr + p)); }
  __device__ __forceinline__ SF64Arr lightState() const { return SF64Arr{wa(L.oLight)}; }
  // ---- HBM/L2-resident parts of the blob
  __device__ __forceinline__ double* ctrl(int k) { return reinterpret_cast<double*>(blob + L.oCtrl) + 4 * k; }
  __device__ __forceinline__ float* manifoldRec(int i) { return blob + L.oMan + MR_WORDS * i; }
  // cached TOI alpha per contact (b2Contact::m_toi): lives in the record region, which is free outside solve()
  __device__ __forceinline__ SU32 toiAlpha(int i) const { return SU32{wa(L.sRec + 3 * L.Kmax + 8 + i)}; }
  // general-constraint records: in the free part of the shared-memory record region when they fit (they almost
  // always do), else in the blob (HBM/L2).  genBase is a generic pointer either way; the records are only ever
  // touched by the one lane that owns them.
  __device__ __forceinline__ float* smemGeneric(int word) const {
    return reinterpret_cast<float*>(__cvta_shared_to_generic((size_t)wa(word)));
  }
  __device__ __forceinline__ float& pool(int f, int q) { return genBase[GR_WORDS * q + f]; }
  __device__ __forceinline__ uint32_t& poolu(int f, int q) { return reinterpret_cast<uint32_t*>(genBase)[GR_WORDS * q + f]; }
  __device__ __forceinline__ float& gw(int q, int w) { return genBase[GR_WORDS * q + w]; }

  __device__ __forceinline__ Xf bodyXf(int b) {
    float4 x = xf4(b);
    Xf t;
    t.p = mk(x.x, x.y);
    t.q.s = x.z;
    t.q.c = x.w;
    return t;
  }
  __device__ __forceinline__ bool awake(int b) { return (f2u(vel4(b).get(3)) & BF_AWAKE) != 0u; }
  // b2Body::SetAwake(true): only acts on sleeping bodies
  __device__ __forceinline__ void wake(int b) {
    if (b == S) return;
    uint32_t f = f2u(vel4(b).get(3));
    if ((f & BF_AWAKE) == 0u) {
      vel4(b).set(3, u2f(f | BF_AWAKE));
      pos4(b).set(3, 0.0f);
    }
  }

  // ------------------------------------------------------------------------- state I/O
  __device__ __forceinline__ void loadState() {
    const float4* src = reinterpret_cast<const float4*>(blob);
    const int n4 = L.stateWords >> 2;
#pragma unroll 1
    for (int i = g.lane; i < n4; i += LPE) sts_f4(sa + 16u * (uint32_t)i, src[i]);
    g.usync();
  }
  __device__ __forceinline__ void storeState() {
    g.usync();
    float4* dst = reinterpret_cast<float4*>(blob);
    const int n4 = L.stateWords >> 2;
#pragma unroll 1
    for (int i = g.lane; i < n4; i += LPE) dst[i] = lds_f4(sa + 16u * (uint32_t)i);
    if (g.lane == 0) {
      unsigned long long* c = reinterpret_cast<unsigned long long*>(blob + L.oCnt);
      c[KB_CNT_SUBSTEPS] += nSub;
      c[KB_CNT_CONTACTS] += nCon;
      c[KB_CNT_POINTS] += nPts;
      c[KB_CNT_LEVELS] += nLvl;
      c[KB_CNT_POS_ITERS] += nPit;
      c[KB_CNT_TOI_EVENTS] += nToi;
      c[KB_CNT_PAIR_TESTS] += nTests;
      c[KB_CNT_ISLANDS] += nIsl;
    }
  }
  // scratch that is constant for the launch: body constants, static-table slot, proxy->body map,
  // adjacency masks of the persistent contact list
  __device__ __forceinline__ void initScratch() {
#pragma unroll 1
    for (int b = g.lane; b <= L.B; b += LPE) {
      if (b < L.B) {
        const BodyConst* c = bc + b;
        bc4(b) = make_float4(__ldg(&c->invMass), __ldg(&c->invI), __ldg(&c->lcx), __ldg(&c->lcy));
        sts_u8(wa(L.sBk) + (uint32_t)b, (uint32_t)__ldg(&c->kind));
        // b2Island::Solve damping factors (SimplePhototaxisKilobot's linearDamping = 0, lib/kilobot.py:203, is
        // folded into the template)
        const float h = L.dt, ld = __ldg(&c->linearDamping), ad = __ldg(&c->angularDamping);
        damp(b) = L.dampingMode == 0 ? make_float2(1.0f / (1.0f + h * ld), 1.0f / (1.0f + h * ad))
                                     : make_float2(b2clamp(1.0f - h * ld, 0.0f, 1.0f), b2clamp(1.0f - h * ad, 0.0f, 1.0f));
      } else {
        bc4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        pos4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        vel4(b) = make_float4(0.0f, 0.0f, 0.0f, u2f(BF_AWAKE));
        xf4(b) = make_float4(0.0f, 0.0f, 0.0f, 1.0f);
        sweep4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      }
    }
#pragma unroll 1
    for (int p = g.lane; p < L.P; p += LPE) {
      sts_u8(wa(L.sPb) + (uint32_t)p, (uint32_t)__ldg(&px[p].body));
      sts_u8(wa(L.sPt) + (uint32_t)p, (uint32_t)__ldg(&px[p].type) | (__ldg(&px[p].friction) == 0.0f ? 4u : 0u) |
                                          (__ldg(&px[p].restitution) == 0.0f ? 8u : 0u));
      sts_f32(wa(L.sPr + p), __ldg(&px[p].radius));
    }
#pragma unroll 1
    for (int p = g.lane; p < 2 * L.P; p += LPE) word(L.sAdj + p) = 0u;
#pragma unroll 1
    for (int w = g.lane; w < LC_WORDS * L.numLights; w += LPE)
      word(L.sLc + w) = __ldg(reinterpret_cast<const uint32_t*>(lights) + w);
    g.usync();
    const int nC = (int)hdr(H_NC);
#pragma unroll 1
    for (int i = g.lane; i < nC; i += LPE) {
      const uint32_t w = cw(i);
      const int pa = CW_PA(w), pb = CW_PB(w);
      adj(pa, pb >> 5).atomOr(1u << (pb & 31));
      adj(pb, pa >> 5).atomOr(1u << (pa & 31));
    }
    g.usync();
  }

  // --------------------------------------------------------------------------- narrowphase
  __device__ __forceinline__ void evaluate(Manifold& m, int pa, int pb, int bA, int bB) {
    const ProxyConst* A = px + pa;
    const ProxyConst* Bp = px + pb;
    const int tA = ptype(pa), tB = ptype(pb);
    const Xf xfA = bodyXf(bA), xfB = bodyXf(bB);
    // every contact of a kilobot is one of the three inlined cases: their manifold stays in registers.  The
    // polygon cases (object against object / table) run out of line on a temporary, the only manifold whose
    // address is ever taken (local memory costs an L2 round trip here: shared memory takes most of the L1).
    if (tB == SHAPE_CIRCLE) {
      if (tA == SHAPE_CIRCLE) collide_circles(m, pradius(pa), xfA, pradius(pb), xfB);
      else if (tA == SHAPE_POLYGON) collide_polygon_circle(m, A, xfA, pradius(pb), xfB);
      else collide_edge_circle(m, A, xfA, pradius(pb), xfB);
    } else {
      Manifold t;
      t.pointCount = 0;
      t.type = 0;
      t.lnx = t.lny = t.lpx = t.lpy = 0.0f;
      t.px[0] = t.py[0] = t.px[1] = t.py[1] = 0.0f;
      t.id[0] = t.id[1] = 0u;
      if (tA == SHAPE_POLYGON) collide_polygons(t, A, xfA, Bp, xfB);
      else collide_edge_polygon(t, A, xfA, Bp, xfB);
      m.pointCount = t.pointCount;
      m.type = t.type;
      m.lnx = t.lnx; m.lny = t.lny; m.lpx = t.lpx; m.lpy = t.lpy;
      m.px[0] = t.px[0]; m.py[0] = t.py[0]; m.px[1] = t.px[1]; m.py[1] = t.py[1];
      m.id[0] = t.id[0]; m.id[1] = t.id[1];
    }
  }

  // b2Contact::Update for contact i (this lane).  Returns true if touching changed.
  __device__ __forceinline__ bool updateContact(int i) {
    uint32_t w = cw(i);
    const int pa = CW_PA(w), pb = CW_PB(w);
    const int bA = pbody(pa), bB = pbody(pb);
    const int oldPC = (w & CI_PC_MASK) >> CI_PC_SHIFT;
    const bool wasTouching = (w & CI_TOUCHING) != 0u;
    Manifold m;
    m.pointCount = 0;
    m.type = 0;
    m.lnx = m.lny = m.lpx = m.lpy = 0.0f;
    m.px[0] = m.py[0] = m.px[1] = m.py[1] = 0.0f;
    m.id[0] = m.id[1] = 0u;
    evaluate(m, pa, pb, bA, bB);
    const bool touching = m.pointCount > 0;
    float* rec = manifoldRec(i);
    if (touching) {
      m.ni[0] = m.ni[1] = m.ti[0] = m.ti[1] = 0.0f;
      if (oldPC > 0) {
        const float4 r1 = reinterpret_cast<const float4*>(rec)[1];  // p0x p0y p0n p0t
        const float4 r2 = reinterpret_cast<const float4*>(rec)[2];  // p0id p1x p1y p1n
        const float4 r3 = reinterpret_cast<const float4*>(rec)[3];  // p1t p1id type pad
        const uint32_t oid0 = f2u(r2.x), oid1 = f2u(r3.y);
        for (int k = 0; k < m.pointCount; ++k) {
          const uint32_t id2 = k == 0 ? m.id[0] : m.id[1];
          float ni = 0.0f, ti = 0.0f;
          if (oid0 == id2) {
            ni = r1.z;
            ti = r1.w;
          } else if (oldPC > 1 && oid1 == id2) {
            ni = r2.w;
            ti = r3.x;
          }
          if (k == 0) { m.ni[0] = ni; m.ti[0] = ti; }
          else { m.ni[1] = ni; m.ti[1] = ti; }
        }
      }
      float4* o = reinterpret_cast<float4*>(rec);
      o[0] = make_float4(m.lnx, m.lny, m.lpx, m.lpy);
      o[1] = make_float4(m.px[0], m.py[0], m.ni[0], m.ti[0]);
      o[2] = make_float4(u2f(m.id[0]), m.px[1], m.py[1], m.ni[1]);
      o[3] = make_float4(m.ti[1], u2f(m.id[1]), u2f((uint32_t)m.type | ((uint32_t)m.pointCount << 8)), 0.0f);
    }
    w |= CI_ENABLED;
    w = touching ? (w | CI_TOUCHING) : (w & ~CI_TOUCHING);
    w = (w & ~CI_PC_MASK) | ((uint32_t)m.pointCount << CI_PC_SHIFT);
    cw(i) = w;
    return touching != wasTouching;
  }

  // b2ContactManager::Collide.  World-list order is descending array index; a sleeping pair is
  // only visited if an earlier (higher index) contact woke one of its bodies (see DESIGN.md).
  // Written in warp-uniform style: every lane group of the warp walks the same chunks and passes (the trip counts
  // are the warp's maxima), groups that have nothing left to do run them empty, and the votes / barriers are the
  // full-mask u-variants (outside uniform mode they are the group's own).
  __device__ __forceinline__ void collide() {
    const int nC = (int)hdr(H_NC);
    if (!g.uany(nC != 0)) return;
    // any sleeping dynamic body?
    bool sleepy = false;
#pragma unroll 1
    for (int b = g.lane; b < L.B; b += LPE) sleepy |= !awake(b);
    const uint32_t sleepyMask = g.uballot(sleepy);   // every lane votes (no short-circuit around a full-mask vote)
    const bool anyAsleep = nC != 0 && sleepyMask != 0u;
    const bool anyAsleepU = g.uany(anyAsleep);
    // stk(b) doubles as wakeAt[b]: per body, the highest contact index that woke it
    if (anyAsleep) {
#pragma unroll 1
      for (int b = g.lane; b <= L.B; b += LPE) stk(b) = awake(b) ? 0x7FFFFFFF : -1;
    }
    if (anyAsleepU) g.usync();
    bool anyDestroyed = false;
    // chunks from the top: a wake-up caused by a contact reaches every lower-index contact of later chunks in
    // the same pass; another pass is only needed after a pass that woke somebody
    const int top = g.umax((nC + LPE - 1) / LPE) * LPE - LPE;
    for (int pass = 0;; ++pass) {
      bool woke = false;
#pragma unroll 1
      for (int base = top; base >= 0; base -= LPE) {
        const int i = base + g.lane;
        bool doit = false;
        int pa = 0, pb = 0, bA = S, bB = S;
        uint32_t w = 0u;
        if (i < nC && (pass == 0 || anyAsleep)) {
          w = cw(i);
          if ((w & CI_DONE) == 0u) {
            pa = CW_PA(w);
            pb = CW_PB(w);
            bA = pbody(pa);
            bB = pbody(pb);
            if (!anyAsleep) {
              doit = true;
            } else {
              const bool actA = bA != S && (int32_t)stk(bA) > i;
              const bool actB = bB != S && (int32_t)stk(bB) > i;
              doit = actA || actB;
            }
          }
        }
        if (doit) {
          const float4 fa = fat4(pa), fb = fat4(pb);
          // b2TestOverlap
          const bool overlap = !(fb.x - fa.z > 0.0f || fb.y - fa.w > 0.0f || fa.x - fb.z > 0.0f || fa.y - fb.w > 0.0f);
          bool wakeEvent;
          if (!overlap) {
            wakeEvent = (w & CI_PC_MASK) != 0u;
            cw(i) = w | CI_DESTROY | (anyAsleep ? CI_DONE : 0u);
            adj(pa, pb >> 5).atomAnd(~(1u << (pb & 31)));
            adj(pb, pa >> 5).atomAnd(~(1u << (pa & 31)));
            anyDestroyed = true;
          } else {
            wakeEvent = updateContact(i);
            if (anyAsleep) cw(i) |= CI_DONE;
          }
          if (wakeEvent && anyAsleep) {
            if (bA != S) stk(bA).atomMax(i);
            if (bB != S) stk(bB).atomMax(i);
            woke = true;
          }
        }
        if (anyAsleepU) g.usync();
      }
      if (!anyAsleepU) break;
      const uint32_t wokeMask = g.uballot(woke);
      const bool again = wokeMask != 0u && anyAsleep;
      if (!g.uany(again)) break;
    }
    g.usync();
    if (anyAsleep) {
#pragma unroll 1
      for (int b = g.lane; b < L.B; b += LPE)
        if ((int32_t)stk(b) >= 0) wake(b);
    }
    if (anyAsleepU) g.usync();
    // clear DONE marks; stable compaction if anything was destroyed
    const bool compact = g.uballot(anyDestroyed) != 0u;
    if (!g.uany(compact || anyAsleep)) return;
    int out = 0;
    const int nCU = g.umax(nC);
#pragma unroll 1
    for (int base = 0; base < nCU; base += LPE) {
      const int i = base + g.lane;
      uint32_t w = 0u;
      bool keep = false;
      if (i < nC) {
        w = cw(i);
        keep = (w & CI_DESTROY) == 0u;
        w &= ~(CI_DONE | CI_DESTROY);
      }
      const uint32_t m = g.uballot(keep);
      const int dst = compact ? out + __popc(m & g.lt()) : i;
      float4 r0, r1, r2, r3;
      const bool moveRec = keep && dst != i && (w & CI_PC_MASK) != 0u;
      if (moveRec) {
        const float4* rec = reinterpret_cast<const float4*>(manifoldRec(i));
        r0 = rec[0]; r1 = rec[1]; r2 = rec[2]; r3 = rec[3];
      }
      g.usync();
      if (keep) {
        cw(dst) = w;
        if (moveRec) {
          float4* rec = reinterpret_cast<float4*>(manifoldRec(dst));
          rec[0] = r0; rec[1] = r1; rec[2] = r2; rec[3] = r3;
        }
      }
      out += __popc(m);
      g.usync();
    }
    if (compact) {
      if (g.lane == 0) hdr(H_NC) = (uint32_t)out;
    }
    g.usync();
  }

  // ------------------------------------------------------------------------------ solver
  struct VelBody {
    V2 v;
    float w;
  };

  // ---- simple constraints: one manifold point, no friction, no restitution, fixture B a circle
  // (every contact of a kilobot).  Two float4 records per schedule entry, resident in shared memory:
  //   velocity phase: rec[2e] = (normal.x, normal.y, normalMass, normalImpulse), rec[2e+1] = (rA.x, rA.y, rB.x, rB.y)
  //   position phase: rec[2e] = (localNormal, localPoint),                       rec[2e+1] = (radiusA, radiusB, type, -)
  // b2ContactSolver ctor + InitializeVelocityConstraints
  __device__ __forceinline__ void initSimple(int e, int ci, uint32_t item) {
    const int bA = IT_BA(item), bB = IT_BB(item);
    const uint32_t w = cw(ci);
    const int pa = CW_PA(w), pb = CW_PB(w);
    const float4* rec = reinterpret_cast<const float4*>(manifoldRec(ci));
    const float4 r0 = rec[0], r1 = rec[1];
    const int type = (int)(f2u(manifoldRec(ci)[MR_TYPE]) & 0xFFu);
    const float radiusA = pradius(pa), radiusB = pradius(pb);
    const float4 cA4 = pos4(bA), cB4 = pos4(bB);
    const float4 kA = bc4(bA), kB = bc4(bB);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    const V2 cA = mk(cA4.x, cA4.y), cB = mk(cB4.x, cB4.y);
    // xf from (c, a): q == the body's current xf.q (b2Rot::Set(sweep.a) is what produced it)
    Xf xfA, xfB;
    const float4 xa = xf4(bA), xb = xf4(bB);
    xfA.q.s = xa.z; xfA.q.c = xa.w;
    xfB.q.s = xb.z; xfB.q.c = xb.w;
    xfA.p = cA - rmul(xfA.q, mk(kA.z, kA.w));
    xfB.p = cB - rmul(xfB.q, mk(kB.z, kB.w));
    // b2WorldManifold::Initialize
    V2 normal, pt;
    const V2 lp = mk(r0.z, r0.w), ln = mk(r0.x, r0.y);
    const V2 mp0 = mk(r1.x, r1.y);
    if (type == MANIFOLD_CIRCLES) {
      normal = mk(1.0f, 0.0f);
      V2 pointA = xmul(xfA, lp);
      V2 pointB = xmul(xfB, mp0);
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
      V2 clipPoint = xmul(xfB, mp0);
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
    rec4(2 * e) = make_float4(normal.x, normal.y, nMass, r1.z);  // warm start: dtRatio (== 1) * normalImpulse
    rec4(2 * e + 1) = make_float4(rA.x, rA.y, rB.x, rB.y);
  }

  // b2ContactSolver::WarmStart
  __device__ __forceinline__ void warmStartSimple(int e, uint32_t item) {
    const int bA = IT_BA(item), bB = IT_BB(item);
    const float4 r0 = rec4(2 * e), r1 = rec4(2 * e + 1);
    const float4 kA = bc4(bA), kB = bc4(bB);
    float4 vA = vel4(bA), vB = vel4(bB);
    const V2 normal = mk(r0.x, r0.y);
    const V2 tangent = cross(normal, 1.0f);
    const V2 rA = mk(r1.x, r1.y), rB = mk(r1.z, r1.w);
    const V2 P = r0.w * normal + 0.0f * tangent;
    vA.z -= kA.y * cross(rA, P);
    vA.x = vA.x - kA.x * P.x;
    vA.y = vA.y - kA.x * P.y;
    vB.z += kB.y * cross(rB, P);
    vB.x = vB.x + kB.x * P.x;
    vB.y = vB.y + kB.x * P.y;
    vel4(bA) = vA;  // the static slot receives +0 velocities (invMass = invI = 0): harmless
    vel4(bB) = vB;
  }

  // b2ContactSolver::SolveVelocityConstraints (the tangent row contributes exactly zero: friction == 0)
  __device__ __forceinline__ void solveVelocitySimple(int e, uint32_t item) {
    const int bA = IT_BA(item), bB = IT_BB(item);
    const float4 r0 = rec4(2 * e), r1 = rec4(2 * e + 1);
    const float4 kA = bc4(bA), kB = bc4(bB);
    float4 a4 = vel4(bA), b4 = vel4(bB);
    const V2 normal = mk(r0.x, r0.y);
    const V2 rA0 = mk(r1.x, r1.y), rB0 = mk(r1.z, r1.w);
    const V2 Av = mk(a4.x, a4.y), Bv = mk(b4.x, b4.y);
    V2 dv = Bv + cross(b4.z, rB0) - Av - cross(a4.z, rA0);
    float vn = dot(dv, normal);
    float ni = r0.w;
    float lambda = -r0.z * (vn - 0.0f);
    float newImpulse = b2max(ni + lambda, 0.0f);
    lambda = newImpulse - ni;
    V2 P = lambda * normal;
    const V2 Av2 = Av - kA.x * P;
    a4.z -= kA.y * cross(rA0, P);
    const V2 Bv2 = Bv + kB.x * P;
    b4.z += kB.y * cross(rB0, P);
    a4.x = Av2.x; a4.y = Av2.y;
    b4.x = Bv2.x; b4.y = Bv2.y;
    vel4(bA) = a4;
    vel4(bB) = b4;
    rec4(2 * e).set(3, newImpulse);
  }

  // the same two with the entry's records (r0, r1), inverse masses kk = (mA, iA, mB, iB) and body rows in registers
  __device__ __forceinline__ void warmStartCached(SF4 rowA, SF4 rowB, const float4& r0, const float4& r1, const float4& kk) {
    float4 vA = rowA, vB = rowB;
    const V2 normal = mk(r0.x, r0.y);
    const V2 tangent = cross(normal, 1.0f);
    const V2 rA = mk(r1.x, r1.y), rB = mk(r1.z, r1.w);
    const V2 P = r0.w * normal + 0.0f * tangent;
    vA.z -= kk.y * cross(rA, P);
    vA.x = vA.x - kk.x * P.x;
    vA.y = vA.y - kk.x * P.y;
    vB.z += kk.w * cross(rB, P);
    vB.x = vB.x + kk.z * P.x;
    vB.y = vB.y + kk.z * P.y;
    rowA = vA;
    rowB = vB;
  }
  __device__ __forceinline__ float solveVelocityCached(SF4 rowA, SF4 rowB, const float4& r0, const float4& r1, const float4& kk) {
    float4 a4 = rowA, b4 = rowB;
    const V2 normal = mk(r0.x, r0.y);
    const V2 rA0 = mk(r1.x, r1.y), rB0 = mk(r1.z, r1.w);
    const V2 Av = mk(a4.x, a4.y), Bv = mk(b4.x, b4.y);
    V2 dv = Bv + cross(b4.z, rB0) - Av - cross(a4.z, rA0);
    float vn = dot(dv, normal);
    float ni = r0.w;
    float lambda = -r0.z * (vn - 0.0f);
    float newImpulse = b2max(ni + lambda, 0.0f);
    lambda = newImpulse - ni;
    V2 P = lambda * normal;
    const V2 Av2 = Av - kk.x * P;
    a4.z -= kk.y * cross(rA0, P);
    const V2 Bv2 = Bv + kk.z * P;
    b4.z += kk.w * cross(rB0, P);
    a4.x = Av2.x; a4.y = Av2.y;
    b4.x = Bv2.x; b4.y = Bv2.y;
    rowA = a4;
    rowB = b4;
    return newImpulse;
  }

  // b2ContactSolver::StoreImpulses, then re-purpose the records for the position solver
  __device__ __forceinline__ void storeSimple(int e, int ci, uint32_t item) {
    float* rec = manifoldRec(ci);
    rec[MR_P0N] = rec4(2 * e).get(3);
    const float4 r0 = reinterpret_cast<const float4*>(rec)[0];
    const uint32_t tp = f2u(rec[MR_TYPE]);
    const uint32_t w = cw(ci);
    rec4(2 * e) = r0;
    rec4(2 * e + 1) = make_float4(pradius(CW_PA(w)), pradius(CW_PB(w)), u2f(tp & 0xFFu), 0.0f);
    // the position sweeps decide once per solve, not once per row-step, whether this entry is the
    // kilobot-against-kilobot case of solvePositionSimple (the predicate is copied from there)
    const int bA = IT_BA(item), bB = IT_BB(item);
    const float4 kA = bc4(bA), kB = bc4(bB);
    const bool trigA = bA != S && ((int)(tp & 0xFFu) != MANIFOLD_CIRCLES || r0.z != 0.0f || r0.w != 0.0f ||
                                   kA.z != 0.0f || kA.w != 0.0f);
    const bool trigB = bB != S && (kB.z != 0.0f || kB.w != 0.0f);
    if ((int)(tp & 0xFFu) == MANIFOLD_CIRCLES && bA != S && !trigA && !trigB) ent(e) = item | IT_FAST;
  }

  // solvePositionSimple for an IT_FAST entry: the same operations in the same order, without the case analysis
  __device__ __forceinline__ bool solvePositionFast(int e, uint32_t item) {
    const int bA = IT_BA(item), bB = IT_BB(item);
    const float4 r1 = rec4(2 * e + 1);
    const float4 kA = bc4(bA), kB = bc4(bB);
    const float4 pA4 = pos4(bA), pB4 = pos4(bB);
    float4 a1, b1;
    bool moved, bad = false;
    bool ok = kb_position_pair_t<false>(pA4, pB4, r1.x, r1.y, kA.x, kA.y, kB.x, kB.y, KB_BAUMGARTE, -3.0f * KB_LINEAR_SLOP, true, a1,
                                        b1, moved, bad);
    if (moved) {
      pos4(bA) = a1;
      if (bB != S) pos4(bB) = b1;
    }
    if (__builtin_expect(bad, 0)) {   // (off the dependent chain: the rows are stored already)
      ok = kb_position_pair_cold(pos4(bA).a, bB != S ? pos4(bB).a : 0u, pA4, pB4, r1.x, r1.y, kA.x, kA.y, kB.x, kB.y, KB_BAUMGARTE,
                                 -3.0f * KB_LINEAR_SLOP, true);
    }
    return ok;
  }

  // one constraint of b2ContactSolver::SolvePositionConstraints.  Returns false if the separation is
  // below -3 * linearSlop (island not yet solved).
  __device__ __forceinline__ bool solvePositionSimple(int e, uint32_t item) {
    const int bA = IT_BA(item), bB = IT_BB(item);
    const float4 r0 = rec4(2 * e), r1 = rec4(2 * e + 1);
    const float4 kA = bc4(bA), kB = bc4(bB);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    const V2 lcA = mk(kA.z, kA.w), lcB = mk(kB.z, kB.w);
    float4 pA4 = pos4(bA), pB4 = pos4(bB);
    V2 cA = mk(pA4.x, pA4.y), cB = mk(pB4.x, pB4.y);
    float aA = pA4.z, aB = pB4.z;
    const V2 ln = mk(r0.x, r0.y);
    const V2 lp = mk(r0.z, r0.w);
    const float radiusA = r1.x, radiusB = r1.y;
    const int type = (int)f2u(r1.z);
    // a rotation is only needed where it multiplies something non-zero (0 * finite == 0 exactly)
    const bool trigA = bA != S && (type != MANIFOLD_CIRCLES || lp.x != 0.0f || lp.y != 0.0f || lcA.x != 0.0f ||
                                   lcA.y != 0.0f);
    const bool trigB = bB != S && (lcB.x != 0.0f || lcB.y != 0.0f);
    const V2 mpj = mk(0.0f, 0.0f);
    V2 normal, point;
    float separation;
    if (type == MANIFOLD_CIRCLES && bA != S && !trigA && !trigB) {
      // kilobot against kilobot: local centres and local points are all zero, so xf.p == c and
      // b2Mul(xf, 0) == c exactly (up to the sign of a zero, which no later operation can observe).
      // (bA == S with e_circles is a chain-vertex contact: its local point is the vertex, not zero.)
      normal = cB - cA;
      normalize(normal);
      point = 0.5f * (cA + cB);
      separation = dot(cB - cA, normal) - radiusA - radiusB;
    } else {
      Xf xfA, xfB;
      if (trigA) xfA.q = rot_set(aA);
      else { xfA.q.s = 0.0f; xfA.q.c = 1.0f; }
      if (trigB) xfB.q = rot_set(aB);
      else { xfB.q.s = 0.0f; xfB.q.c = 1.0f; }
      xfA.p = cA - rmul(xfA.q, lcA);
      xfB.p = cB - rmul(xfB.q, lcB);
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
    const bool ok = separation >= -3.0f * KB_LINEAR_SLOP;
    const float C = b2clamp(KB_BAUMGARTE * (separation + KB_LINEAR_SLOP), -KB_MAX_LINEAR_CORRECTION, 0.0f);
    // C == 0 (not penetrating beyond the slop): the impulse is -0 / K and moves nothing
    if (C == 0.0f) return ok;
    const V2 rA = point - cA;
    const V2 rB = point - cB;
    const float rnA = cross(rA, normal);
    const float rnB = cross(rB, normal);
    const float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
    const float impulse = K > 0.0f ? -C / K : 0.0f;
    const V2 P = impulse * normal;
    cA = cA - mA * P;
    aA -= iA * cross(rA, P);
    cB = cB + mB * P;
    aB += iB * cross(rB, P);
    if (bA != S) {
      pA4.x = cA.x; pA4.y = cA.y; pA4.z = aA;
      pos4(bA) = pA4;
    }
    if (bB != S) {
      pB4.x = cB.x; pB4.y = cB.y; pB4.z = aB;
      pos4(bB) = pB4;
    }
    return ok;
  }

  // ---- general constraints (two manifold points, friction or restitution: object-object and
  // object-table contacts, and the TOI mini-island).  Records live in HBM/L2 (GR_WORDS words each);
  // one lane owns a record for the whole solve, so no cross-lane visibility is needed.
  // b2ContactSolver ctor + InitializeVelocityConstraints for general slot q.  fresh == true is the
  // TOI island variant: rotations rebuilt from the (corrected) angles, no warm starting.
  __device__ __forceinline__ void initGeneral(int q, int ci, int bA, int bB, uint32_t aux, bool fresh) {
    const uint32_t w = cw(ci);
    const int pa = CW_PA(w), pb = CW_PB(w);
    const float4* rec = reinterpret_cast<const float4*>(manifoldRec(ci));
    const float4 r0 = rec[0], r1 = rec[1], r2 = rec[2], r3 = rec[3];
    const uint32_t tp = f2u(r3.z);
    const int type = tp & 0xFF, pointCount = (tp >> 8) & 0xFF;
    const float radiusA = pradius(pa), radiusB = pradius(pb);
    const float4 cA4 = pos4(bA), cB4 = pos4(bB);
    const float4 vA4 = vel4(bA), vB4 = vel4(bB);
    const float4 kA = bc4(bA), kB = bc4(bB);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    const V2 cA = mk(cA4.x, cA4.y), cB = mk(cB4.x, cB4.y);
    const V2 vA = mk(vA4.x, vA4.y), vB = mk(vB4.x, vB4.y);
    const float wA = vA4.z, wB = vB4.z;
    Xf xfA, xfB;
    {
      if (fresh) {
        xfA.q = rot_set(cA4.z);
        xfB.q = rot_set(cB4.z);
      } else {
        const float4 xa = xf4(bA), xb = xf4(bB);
        xfA.q.s = xa.z; xfA.q.c = xa.w;
        xfB.q.s = xb.z; xfB.q.c = xb.w;
      }
      xfA.p = cA - rmul(xfA.q, mk(kA.z, kA.w));
      xfB.p = cB - rmul(xfB.q, mk(kB.z, kB.w));
    }
    // b2WorldManifold::Initialize
    V2 normal, pts[2];
    const V2 lp = mk(r0.z, r0.w), ln = mk(r0.x, r0.y);
    const V2 mp0 = mk(r1.x, r1.y), mp1 = mk(r2.y, r2.z);
    if (type == MANIFOLD_CIRCLES) {
      normal = mk(1.0f, 0.0f);
      V2 pointA = xmul(xfA, lp);
      V2 pointB = xmul(xfB, mp0);
      if (distsq(pointA, pointB) > KB_EPS * KB_EPS) {
        normal = pointB - pointA;
        normalize(normal);
      }
      V2 a = pointA + radiusA * normal;
      V2 b = pointB - radiusB * normal;
      pts[0] = 0.5f * (a + b);
      pts[1] = pts[0];
    } else if (type == MANIFOLD_FACE_A) {
      normal = rmul(xfA.q, ln);
      V2 planePoint = xmul(xfA, lp);
      for (int k = 0; k < pointCount; ++k) {
        V2 clipPoint = xmul(xfB, k == 0 ? mp0 : mp1);
        V2 a = clipPoint + (radiusA - dot(clipPoint - planePoint, normal)) * normal;
        V2 b = clipPoint - radiusB * normal;
        pts[k] = 0.5f * (a + b);
      }
    } else {
      normal = rmul(xfB.q, ln);
      V2 planePoint = xmul(xfB, lp);
      for (int k = 0; k < pointCount; ++k) {
        V2 clipPoint = xmul(xfA, k == 0 ? mp0 : mp1);
        V2 b = clipPoint + (radiusB - dot(clipPoint - planePoint, normal)) * normal;
        V2 a = clipPoint - radiusA * normal;
        pts[k] = 0.5f * (a + b);
      }
      normal = -normal;
    }
    const float friction = sqrtf(__ldg(&px[pa].friction) * __ldg(&px[pb].friction));
    const float restA = __ldg(&px[pa].restitution), restB = __ldg(&px[pb].restitution);
    const float restitution = restA > restB ? restA : restB;
    const V2 tangent = cross(normal, 1.0f);
    float nMass[2], tMass[2], bias[2];
    V2 rA[2], rB[2];
    for (int k = 0; k < pointCount; ++k) {
      rA[k] = pts[k] - cA;
      rB[k] = pts[k] - cB;
      float rnA = cross(rA[k], normal);
      float rnB = cross(rB[k], normal);
      float kNormal = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
      nMass[k] = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
      float rtA = cross(rA[k], tangent);
      float rtB = cross(rB[k], tangent);
      float kTangent = mA + mB + iA * rtA * rtA + iB * rtB * rtB;
      tMass[k] = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
      bias[k] = 0.0f;
      float vRel = dot(normal, vB + cross(wB, rB[k]) - vA - cross(wA, rA[k]));
      if (vRel < -KB_VELOCITY_THRESHOLD) bias[k] = -restitution * vRel;
    }
    int vcPointCount = pointCount;
    float k11 = 0.0f, k12 = 0.0f, k22 = 0.0f, nm00 = 0.0f, nm01 = 0.0f, nm10 = 0.0f, nm11 = 0.0f;
    if (pointCount == 2) {
      float rn1A = cross(rA[0], normal);
      float rn1B = cross(rB[0], normal);
      float rn2A = cross(rA[1], normal);
      float rn2B = cross(rB[1], normal);
      k11 = mA + mB + iA * rn1A * rn1A + iB * rn1B * rn1B;
      k22 = mA + mB + iA * rn2A * rn2A + iB * rn2B * rn2B;
      k12 = mA + mB + iA * rn1A * rn2A + iB * rn1B * rn2B;
      const float k_maxConditionNumber = 1000.0f;
      if (k11 * k11 < k_maxConditionNumber * (k11 * k22 - k12 * k12)) {
        // b2Mat22::GetInverse with ex = (k11, k12), ey = (k12, k22)
        float a = k11, b = k12, c = k12, d = k22;
        float det = a * d - b * c;
        if (det != 0.0f) det = 1.0f / det;
        nm00 = det * d;    // ex.x
        nm01 = -det * b;   // ey.x
        nm10 = -det * c;   // ex.y
        nm11 = det * a;    // ey.y
      } else {
        vcPointCount = 1;
      }
    }
    poolu(PF_IDX, q) = (uint32_t)bA | ((uint32_t)bB << 8) | ((uint32_t)vcPointCount << 16) | ((uint32_t)type << 24) |
                       ((uint32_t)pointCount << 28);
    poolu(PF_AUX, q) = aux;
    pool(PF_NX, q) = normal.x;
    pool(PF_NY, q) = normal.y;
    pool(PF_RAX, q) = rA[0].x;
    pool(PF_RAY, q) = rA[0].y;
    pool(PF_RBX, q) = rB[0].x;
    pool(PF_RBY, q) = rB[0].y;
    pool(PF_NMASS, q) = nMass[0];
    pool(PF_NIMP, q) = fresh ? 0.0f : r1.z;  // warm start: dtRatio (== 1) * normalImpulse
    gw(q, 10) = tMass[0];
    gw(q, 11) = fresh ? 0.0f : r1.w;  // tangentImpulse
    gw(q, 12) = bias[0];
    gw(q, 13) = friction;
    gw(q, 14) = k11;
    gw(q, 15) = k12;
    gw(q, 16) = k22;
    gw(q, 17) = nm00;
    gw(q, 18) = nm01;
    gw(q, 19) = nm11;
    if (pointCount == 2) {
      gw(q, 20) = rA[1].x;
      gw(q, 21) = rA[1].y;
      gw(q, 22) = rB[1].x;
      gw(q, 23) = rB[1].y;
      gw(q, 24) = nMass[1];
      gw(q, 25) = fresh ? 0.0f : r2.w;  // p1 normalImpulse
      gw(q, 26) = tMass[1];
      gw(q, 27) = fresh ? 0.0f : r3.x;  // p1 tangentImpulse
      gw(q, 28) = bias[1];
    }
    gw(q, 29) = nm10;
  }

  __device__ __forceinline__ void loadVel(int b, VelBody& o) {
    float4 v = vel4(b);
    o.v = mk(v.x, v.y);
    o.w = v.z;
  }
  __device__ __forceinline__ void storeVel(int b, const VelBody& o) {
    if (b == S) return;
    vel4(b).set(0, o.v.x);
    vel4(b).set(1, o.v.y);
    vel4(b).set(2, o.w);
  }

  // b2ContactSolver::WarmStart for one general constraint
  __device__ __forceinline__ void warmStartGeneral(int q) {
    const uint32_t idx = poolu(PF_IDX, q);
    const int bA = idx & 0xFF, bB = (idx >> 8) & 0xFF;
    const int pointCount = (idx >> 16) & 0xF;
    const float4 kA = bc4(bA), kB = bc4(bB);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    VelBody A, Bv;
    loadVel(bA, A);
    loadVel(bB, Bv);
    const V2 normal = mk(pool(PF_NX, q), pool(PF_NY, q));
    const V2 tangent = cross(normal, 1.0f);
    {
      const V2 rA = mk(pool(PF_RAX, q), pool(PF_RAY, q)), rB = mk(pool(PF_RBX, q), pool(PF_RBY, q));
      const float ni = pool(PF_NIMP, q);
      const float ti = gw(q, 11);
      V2 P = ni * normal + ti * tangent;
      A.w -= iA * cross(rA, P);
      A.v = A.v - mA * P;
      Bv.w += iB * cross(rB, P);
      Bv.v = Bv.v + mB * P;
    }
    if (pointCount == 2) {
      const V2 rA = mk(gw(q, 20), gw(q, 21)), rB = mk(gw(q, 22), gw(q, 23));
      V2 P = gw(q, 25) * normal + gw(q, 27) * tangent;
      A.w -= iA * cross(rA, P);
      A.v = A.v - mA * P;
      Bv.w += iB * cross(rB, P);
      Bv.v = Bv.v + mB * P;
    }
    storeVel(bA, A);
    storeVel(bB, Bv);
  }

  // b2ContactSolver::SolveVelocityConstraints for one general constraint
  __device__ __forceinline__ void solveVelocityGeneral(int q) {
    const uint32_t idx = poolu(PF_IDX, q);
    const int bA = idx & 0xFF, bB = (idx >> 8) & 0xFF;
    const int pointCount = (idx >> 16) & 0xF;
    const float4 kA = bc4(bA), kB = bc4(bB);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    VelBody A, Bv;
    loadVel(bA, A);
    loadVel(bB, Bv);
    const V2 normal = mk(pool(PF_NX, q), pool(PF_NY, q));
    const V2 rA0 = mk(pool(PF_RAX, q), pool(PF_RAY, q)), rB0 = mk(pool(PF_RBX, q), pool(PF_RBY, q));
    const V2 tangent = cross(normal, 1.0f);
    const float friction = gw(q, 13);
    V2 rA1 = rA0, rB1 = rB0;
    if (pointCount == 2) {
      rA1 = mk(gw(q, 20), gw(q, 21));
      rB1 = mk(gw(q, 22), gw(q, 23));
    }
    // tangent rows first
    for (int j = 0; j < pointCount; ++j) {
      const V2 rA = j == 0 ? rA0 : rA1, rB = j == 0 ? rB0 : rB1;
      const float tMass = j == 0 ? gw(q, 10) : gw(q, 26);
      const float nImp = j == 0 ? pool(PF_NIMP, q) : gw(q, 25);
      float& tImp = j == 0 ? gw(q, 11) : gw(q, 27);
      V2 dv = Bv.v + cross(Bv.w, rB) - A.v - cross(A.w, rA);
      float vt = dot(dv, tangent) - 0.0f;
      float lambda = tMass * (-vt);
      float maxFriction = friction * nImp;
      float newImpulse = b2clamp(tImp + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - tImp;
      tImp = newImpulse;
      V2 P = lambda * tangent;
      A.v = A.v - mA * P;
      A.w -= iA * cross(rA, P);
      Bv.v = Bv.v + mB * P;
      Bv.w += iB * cross(rB, P);
    }
    if (pointCount == 1) {
      V2 dv = Bv.v + cross(Bv.w, rB0) - A.v - cross(A.w, rA0);
      float vn = dot(dv, normal);
      float ni = pool(PF_NIMP, q);
      float lambda = -pool(PF_NMASS, q) * (vn - gw(q, 12));
      float newImpulse = b2max(ni + lambda, 0.0f);
      lambda = newImpulse - ni;
      pool(PF_NIMP, q) = newImpulse;
      V2 P = lambda * normal;
      A.v = A.v - mA * P;
      A.w -= iA * cross(rA0, P);
      Bv.v = Bv.v + mB * P;
      Bv.w += iB * cross(rB0, P);
    } else {
      // block solver
      const float k11 = gw(q, 14), k12 = gw(q, 15), k22 = gw(q, 16);
      const float nm00 = gw(q, 17), nm01 = gw(q, 18), nm10 = gw(q, 29), nm11 = gw(q, 19);
      const float nMass1 = pool(PF_NMASS, q), nMass2 = gw(q, 24);
      V2 a = mk(pool(PF_NIMP, q), gw(q, 25));
      V2 dv1 = Bv.v + cross(Bv.w, rB0) - A.v - cross(A.w, rA0);
      V2 dv2 = Bv.v + cross(Bv.w, rB1) - A.v - cross(A.w, rA1);
      float vn1 = dot(dv1, normal);
      float vn2 = dot(dv2, normal);
      V2 b;
      b.x = vn1 - gw(q, 12);
      b.y = vn2 - gw(q, 28);
      // b -= K a ; K.ex = (k11,k12), K.ey = (k12,k22)
      b = b - mk(k11 * a.x + k12 * a.y, k12 * a.x + k22 * a.y);
      V2 x;
      bool found = false;
      // case 1
      {
        V2 t = mk(nm00 * b.x + nm01 * b.y, nm10 * b.x + nm11 * b.y);
        x = -t;
        if (x.x >= 0.0f && x.y >= 0.0f) found = true;
      }
      if (!found) {  // case 2
        x.x = -nMass1 * b.x;
        x.y = 0.0f;
        vn2 = k12 * x.x + b.y;
        if (x.x >= 0.0f && vn2 >= 0.0f) found = true;
      }
      if (!found) {  // case 3
        x.x = 0.0f;
        x.y = -nMass2 * b.y;
        vn1 = k12 * x.y + b.x;
        if (x.y >= 0.0f && vn1 >= 0.0f) found = true;
      }
      if (!found) {  // case 4
        x.x = 0.0f;
        x.y = 0.0f;
        vn1 = b.x;
        vn2 = b.y;
        if (vn1 >= 0.0f && vn2 >= 0.0f) found = true;
      }
      if (found) {
        V2 d = x - a;
        V2 P1 = d.x * normal;
        V2 P2 = d.y * normal;
        A.v = A.v - mA * (P1 + P2);
        A.w -= iA * (cross(rA0, P1) + cross(rA1, P2));
        Bv.v = Bv.v + mB * (P1 + P2);
        Bv.w += iB * (cross(rB0, P1) + cross(rB1, P2));
        pool(PF_NIMP, q) = x.x;
        gw(q, 25) = x.y;
      }
    }
    storeVel(bA, A);
    storeVel(bB, Bv);
  }

  // b2ContactSolver::StoreImpulses, then re-purpose the record for the position solver
  __device__ __forceinline__ void storeGeneral(int q) {
    const uint32_t idx = poolu(PF_IDX, q);
    const uint32_t aux = poolu(PF_AUX, q);
    const int ci = aux & 0xFFFF;
    const int vcPointCount = (idx >> 16) & 0xF;
    float* rec = manifoldRec(ci);
    rec[MR_P0N] = pool(PF_NIMP, q);
    rec[MR_P0T] = gw(q, 11);
    if (vcPointCount == 2) {
      rec[MR_P1N] = gw(q, 25);
      rec[MR_P1T] = gw(q, 27);
    }
    preparePositionGeneral(q, ci);
  }
  // position data: localNormal, localPoint, radii and both manifold points
  __device__ __forceinline__ void preparePositionGeneral(int q, int ci) {
    const float* rec = manifoldRec(ci);
    const float4 r0 = reinterpret_cast<const float4*>(rec)[0];
    const float4 r1 = reinterpret_cast<const float4*>(rec)[1];
    const float4 r2 = reinterpret_cast<const float4*>(rec)[2];
    const uint32_t w = cw(ci);
    pool(PF_NX, q) = r0.x;
    pool(PF_NY, q) = r0.y;
    pool(PF_RAX, q) = r0.z;
    pool(PF_RAY, q) = r0.w;
    pool(PF_RBX, q) = __ldg(&px[CW_PA(w)].radius);
    pool(PF_RBY, q) = __ldg(&px[CW_PB(w)].radius);
    gw(q, 10) = r1.x;
    gw(q, 11) = r1.y;
    gw(q, 12) = r2.y;
    gw(q, 13) = r2.z;
  }

  // one general constraint of b2ContactSolver::SolvePositionConstraints / SolveTOIPositionConstraints.
  // Returns false if any point's separation is below `limit` (island not yet solved).
  __device__ __forceinline__ bool solvePositionGeneral(int q, float baumgarte, float limit, int toiA, int toiB) {
    const uint32_t idx = poolu(PF_IDX, q);
    const int bA = idx & 0xFF, bB = (idx >> 8) & 0xFF;
    const int type = (idx >> 24) & 0xF;
    const int pointCount = (idx >> 28) & 0xF;
    const float4 kA = bc4(bA), kB = bc4(bB);
    float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    if (toiA >= 0) {
      if (!(bA == toiA || bA == toiB)) { mA = 0.0f; iA = 0.0f; }
      if (!(bB == toiA || bB == toiB)) { mB = 0.0f; iB = 0.0f; }
    }
    const V2 lcA = mk(kA.z, kA.w), lcB = mk(kB.z, kB.w);
    float4 pA4 = pos4(bA), pB4 = pos4(bB);
    V2 cA = mk(pA4.x, pA4.y), cB = mk(pB4.x, pB4.y);
    float aA = pA4.z, aB = pB4.z;
    const V2 ln = mk(pool(PF_NX, q), pool(PF_NY, q));
    const V2 lp = mk(pool(PF_RAX, q), pool(PF_RAY, q));
    const float radiusA = pool(PF_RBX, q), radiusB = pool(PF_RBY, q);
    const bool trigA = bA != S, trigB = bB != S;
    bool ok = true;
    for (int j = 0; j < pointCount; ++j) {
      Xf xfA, xfB;
      if (trigA) xfA.q = rot_set(aA);
      else { xfA.q.s = 0.0f; xfA.q.c = 1.0f; }
      if (trigB) xfB.q = rot_set(aB);
      else { xfB.q.s = 0.0f; xfB.q.c = 1.0f; }
      xfA.p = cA - rmul(xfA.q, lcA);
      xfB.p = cB - rmul(xfB.q, lcB);
      const V2 mpj = j == 0 ? mk(gw(q, 10), gw(q, 11)) : mk(gw(q, 12), gw(q, 13));
      V2 normal, point;
      float separation;
      if (type == MANIFOLD_CIRCLES) {
        V2 pointA = xmul(xfA, lp);
        V2 pointB = xmul(xfB, mpj);
        normal = pointB - pointA;
        normalize(normal);
        point = 0.5f * (pointA + pointB);
        separation = dot(pointB - pointA, normal) - radiusA - radiusB;
      } else if (type == MANIFOLD_FACE_A) {
        normal = rmul(xfA.q, ln);
        V2 planePoint = xmul(xfA, lp);
        V2 clipPoint = xmul(xfB, mpj);
        separation = dot(clipPoint - planePoint, normal) - radiusA - radiusB;
        point = clipPoint;
      } else {
        normal = rmul(xfB.q, ln);
        V2 planePoint = xmul(xfB, lp);
        V2 clipPoint = xmul(xfA, mpj);
        separation = dot(clipPoint - planePoint, normal) - radiusA - radiusB;
        point = clipPoint;
        normal = -normal;
      }
      V2 rA = point - cA;
      V2 rB = point - cB;
      if (!(separation >= limit)) ok = false;
      float C = b2clamp(baumgarte * (separation + KB_LINEAR_SLOP), -KB_MAX_LINEAR_CORRECTION, 0.0f);
      float rnA = cross(rA, normal);
      float rnB = cross(rB, normal);
      float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
      float impulse = K > 0.0f ? -C / K : 0.0f;
      V2 P = impulse * normal;
      cA = cA - mA * P;
      aA -= iA * cross(rA, P);
      cB = cB + mB * P;
      aB += iB * cross(rB, P);
    }
    if (bA != S) {
      pos4(bA).set(0, cA.x); pos4(bA).set(1, cA.y); pos4(bA).set(2, aA);
    }
    if (bB != S) {
      pos4(bB).set(0, cB.x); pos4(bB).set(1, cB.y); pos4(bB).set(2, aB);
    }
    return ok;
  }

  // general slot of schedule entry e (kept in the entry's otherwise unused simple record)
  __device__ __forceinline__ int genSlot(int e) { return (int)lds_u8(wa(L.sGs) + (uint32_t)e); }

  // b2World::Solve
  __device__ __forceinline__ void solve() {
    const int nC = (int)hdr(H_NC);
    const int B = L.B;
    const int KW = L.KW;
    // ---- touching list in world-list order (descending index) and per-body masks over it
#pragma unroll 1
    for (int i = g.lane; i < (B + 1) * KW; i += LPE) word(L.sBmask + i) = 0u;
#pragma unroll 1
    for (int b = g.lane; b <= B; b += LPE) {
      isl(b) = -1;
      lastLvl(b) = 0u;
    }
    g.usync();
    int K = 0;
    const int nCU = g.umax(nC);   // warp-uniform trip count: one full-mask vote serves every lane group of the warp
#pragma unroll 1
    for (int base = 0; base < nCU; base += LPE) {
      const int i = nC - 1 - (base + g.lane);
      bool t = false;
      uint32_t val = 0u;
      int bA = S, bB = S;
      if (i >= 0) {
        const uint32_t w = cw(i);
        t = (w & (CI_TOUCHING | CI_ENABLED)) == (CI_TOUCHING | CI_ENABLED);
        if (t) {
          const int pa = CW_PA(w), pb = CW_PB(w);
          bA = pbody(pa);
          bB = pbody(pb);
          const int pc = (w & CI_PC_MASK) >> CI_PC_SHIFT;
          // mixed friction sqrt(fA * fB) == 0 and mixed restitution max(rA, rB) == 0
          const int fa = pflags(pa), fb = pflags(pb);
          const bool simple = pc == 1 && ((fa | fb) & 4) != 0 && (fa & fb & 8) != 0 && (fb & 3) == SHAPE_CIRCLE;
          val = (uint32_t)i | ((uint32_t)bA << 16) | ((uint32_t)bB << 22) | (simple ? 0u : TL_GEN);
        }
      }
      const uint32_t m = g.uballot(t);
      const int dst = K + __popc(m & g.lt());
      if (t && dst < L.Kmax) {
        tl(dst) = val;
        if (bA != S) bmask(bA, dst >> 5).atomOr(1u << (dst & 31));
        if (bB != S) bmask(bB, dst >> 5).atomOr(1u << (dst & 31));
      }
      K += __popc(m);
    }
    if (K > L.Kmax) {
      if (g.lane == 0) hdr(H_STATUS) |= KB_STATUS_SOLVER_OVERFLOW;
      K = L.Kmax;
    }
#pragma unroll 1
    for (int l = g.lane; l <= K + 1; l += LPE) lvlTab(l) = 0u;
    unsigned long long awakeMask = 0ull;  // awake dynamic bodies (every lane holds the whole mask)
#pragma unroll 1
    for (int bb = 0; bb < B; bb += LPE) {
      const int b = bb + g.lane;
      awakeMask |= (unsigned long long)g.uballot(b < B && awake(b)) << bb;
    }
    g.usync();
    // awake bodies without a touching contact are islands of their own (b2World::Solve seeds them like any other
    // awake body and finds nothing to add): they get their island numbers in parallel below, after the numbers of
    // the islands lane 0 builds.  Island numbers are labels -- nothing depends on their order.
    unsigned long long lonely;
    {
      unsigned long long hasC = 0ull;
#pragma unroll 1
      for (int bb = 0; bb < B; bb += LPE) {
        const int b = bb + g.lane;
        bool c = false;
        if (b < B)
          for (int w4 = 0; w4 < KW; w4 += 4) {
            const uint4 m = lds_u4(wa(L.sBmask + b * KW + w4));
            c |= (m.x | m.y | m.z | m.w) != 0u;
          }
        hasC |= (unsigned long long)g.uballot(c) << bb;
      }
      lonely = awakeMask & ~hasC;
    }
    KB_T(2);
    // ---- lane 0: island DFS (b2World::Solve) in Box2D's order, dependency level of every constraint,
    //      rows, and the level-sorted schedule.  Slot S of bmask collects the contacts already in an island.
    if (g.lane == 0) {
      unsigned long long bflag = 0ull;
      unsigned long long todo = awakeMask & ~lonely;  // awake dynamic bodies with contacts, not in an island yet
      int nOrd = 0, nIslands = 0, maxL = 0;
      while (todo != 0ull) {
        const int seed = 63 - __clzll((long long)todo);  // body list order: newest (highest index) first
        todo &= ~(1ull << seed);
        bflag |= 1ull << seed;
        int sp = 0;
        stk(sp++) = seed;
        while (sp > 0) {
          const int b = stk(--sp);
          isl(b) = nIslands;
          if (((awakeMask >> b) & 1ull) == 0ull) wake(b);
          for (int w4 = 0; w4 < KW; w4 += 4) {
            const uint4 bm = lds_u4(wa(L.sBmask + b * KW + w4));
            const uint4 cf = lds_u4(wa(L.sBmask + S * KW + w4));
            uint32_t mm[4] = {bm.x & ~cf.x, bm.y & ~cf.y, bm.z & ~cf.z, bm.w & ~cf.w};
            if ((mm[0] | mm[1] | mm[2] | mm[3]) == 0u) continue;
            sts_u4(wa(L.sBmask + S * KW + w4), make_uint4(cf.x | mm[0], cf.y | mm[1], cf.z | mm[2], cf.w | mm[3]));
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              uint32_t m = mm[q];
              while (m != 0u) {
                const int t = ((w4 + q) << 5) + __ffs(m) - 1;
                m &= m - 1u;
                const uint32_t tv = tl(t);
                const int bA = (tv >> 16) & 63, bB = (tv >> 22) & 63;
                const int other = bA == b ? bB : bA;
                const uint32_t l = max((uint32_t)lastLvl(bA), (uint32_t)lastLvl(bB)) + 1u;
                lastLvl(bA) = l;
                lastLvl(bB) = l;
                lastLvl(S) = 0u;
                ord(nOrd++) = (uint32_t)t | (l << 10) | ((uint32_t)nIslands << 20);   // 10-bit list index and level
                lvlTab(l) += 1u;
                maxL = max(maxL, (int)l);
                if (other != S && ((bflag >> other) & 1ull) == 0ull) {
                  bflag |= 1ull << other;
                  todo &= ~(1ull << other);
                  stk(sp++) = other;
                }
              }
            }
          }
        }
        ++nIslands;
      }
      // levels -> packed (cursor | first entry << 10 | first row << 20)
      int e0 = 0, row = 0;
      for (int l = 1; l <= maxL; ++l) {
        const int c = (int)lvlTab(l);
        lvlTab(l) = (uint32_t)e0 | ((uint32_t)e0 << 10) | ((uint32_t)row << 20);
        e0 += c;
        row += (c + LPE - 1) / LPE;
      }
      // scatter in constraint order: entries of one level keep Box2D's order
      int nGen = 0;
      for (int p = 0; p < nOrd; ++p) {
        const uint32_t o = ord(p);
        const uint32_t tv = tl(o & 0x3FFu);
        const int l = (o >> 10) & 0x3FF;
        const uint32_t w = lvlTab(l);
        lvlTab(l) = w + 1u;
        const int e = w & 0x3FF, first = (w >> 10) & 0x3FF;
        const int r = (int)(w >> 20) + (e - first) / LPE;
        const bool gen = (tv & TL_GEN) != 0u;
        ent(e) = ((tv >> 16) & 0xFFFu) | ((o >> 20) << 12) | (gen ? IT_GEN : 0u) | ((uint32_t)r << 22);
        entC(e) = (uint16_t)(tv & 0xFFFFu);
        if (gen) {
          if (nGen >= L.Gmax) {
            hdr(H_STATUS) |= KB_STATUS_SOLVER_OVERFLOW;
            nGen = L.Gmax - 1;
          }
          sts_u8(wa(L.sGs) + (uint32_t)e, (uint32_t)nGen++);
        }
      }
      misc(0) = (uint32_t)nOrd;
      misc(1) = (uint32_t)row;
      misc(2) = (uint32_t)nIslands;
      misc(3) = (uint32_t)maxL;
      misc(4) = (uint32_t)nGen;
    }
    g.usync();
    const int nOrd = (int)misc(0), nRows = (int)misc(1), nIslDfs = (int)misc(2);
    const int nIslands = nIslDfs + __popcll(lonely);
#pragma unroll 1
    for (int b = g.lane; b < B; b += LPE)
      if (((lonely >> b) & 1ull) != 0ull) isl(b) = nIslDfs + __popcll(lonely & ((1ull << b) - 1ull));
    const int nRowsU = g.umax(nRows);  // warp-uniform row count: the groups of a warp sweep their rows in lock step
    {
      const int nGen = (int)misc(4);
      genBase = (8 * nOrd + GR_WORDS * nGen <= L.recWords) ? smemGeneric(L.sRec + 8 * nOrd) : blob + L.oGen;
    }
    KB_T(3);
    nIsl += (uint32_t)nIslands;
    nLvl += misc(3);
    // ---- b2Island::Solve: integrate velocities (damping), remember the sweep start
    const float h = L.dt;
#pragma unroll 1
    for (int b = g.lane; b < B; b += LPE) {
      if (isl(b) < 0) continue;
      const float4 p = pos4(b);
      const float4 x = xf4(b);
      sweep4(b) = make_float4(p.x, p.y, p.z, 0.0f);
      oldq(b) = make_float2(x.z, x.w);
      float4 v = vel4(b);
      const float2 df = damp(b);
      v.x *= df.x;
      v.y *= df.x;
      v.z *= df.y;
      vel4(b) = v;
    }
    g.usync();
    // ---- constraints.  Entry e is owned by lane e % LPE for the whole solve.
    {
      uint32_t pts = 0u;
#pragma unroll 1
      for (int e = g.lane; e < nOrd; e += LPE) {
        const uint32_t item = ent(e);
        const int ci = (int)entC(e);
        if ((item & IT_GEN) != 0u) {
          initGeneralNI(*this, genSlot(e), ci, item);
          pts += (cw(ci) & CI_PC_MASK) >> CI_PC_SHIFT;
        } else {
          initSimple(e, ci, item);
          pts += 1u;
        }
      }
      nPts += g.ured_add(pts);
    }
    g.usync();
    KB_T(4);
    // warm start, then velocity iterations: a lane walks its entries in row order.  Its FIRST entry (slot 0: e == lane,
    // the lowest row the lane has) stays in registers for all 1 + velIters passes when it is a simple constraint --
    // records, inverse masses, the two bodies' rows and the accumulated impulse: a row-step of slot 0 is two loads, the
    // arithmetic and two stores.  Measured: C5 (4 lanes per env) 183.5 -> 193.1 M kilobot-steps/s, C3 (32 lanes) 38.6 -> 40.4 M,
    // but C2 (8 lanes: rows that mix slot-0 and second entries run both bodies) 1.035 -> 1.046 ms, so the 8- and 16-lane
    // kernels keep every entry on the ordinary path; folding the two bodies into one (operands selected) lost on all three.
    {
      constexpr bool SLOT0 = LPE == 4 || LPE == 32;
      const uint32_t it0 = (SLOT0 && g.lane < nOrd) ? ent(g.lane) : IT_NONE;
      const bool c0 = SLOT0 && it0 != IT_NONE && (it0 & IT_GEN) == 0u;
      const int row0 = c0 ? IT_ROW(it0) : -1;
      const int kFirst = c0 ? g.lane + LPE : g.lane;   // the entries walked the ordinary way
      float4 q0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), q1 = q0, kk = q0;
      SF4 vA{0u}, vB{0u};
      if (c0) {
        q0 = rec4(2 * g.lane);
        q1 = rec4(2 * g.lane + 1);
        const float4 kA = bc4(IT_BA(it0)), kB = bc4(IT_BB(it0));
        kk = make_float4(kA.x, kA.y, kB.x, kB.y);
        vA = vel4(IT_BA(it0));
        vB = vel4(IT_BB(it0));
      }
      {
        int k = kFirst;
        uint32_t item = k < nOrd ? ent(k) : IT_NONE;
        for (int r = 0; r < nRowsU; ++r) {
          if (r == row0) {
            warmStartCached(vA, vB, q0, q1, kk);
          } else if (IT_ROW(item) == r) {
            const uint32_t cur = item;
            const int kc = k;
            k += LPE;
            item = k < nOrd ? ent(k) : IT_NONE;  // next entry of this lane: fetched while the current one is solved
            if ((cur & IT_GEN) != 0u) warmStartGeneralNI(*this, genSlot(kc));
            else warmStartSimple(kc, cur);
          }
          g.usync();
        }
      }
      for (int it = 0; it < L.velIters; ++it) {
        int k = kFirst;
        uint32_t item = k < nOrd ? ent(k) : IT_NONE;
        for (int r = 0; r < nRowsU; ++r) {
          if (r == row0) {
            q0.w = solveVelocityCached(vA, vB, q0, q1, kk);
          } else if (IT_ROW(item) == r) {
            const uint32_t cur = item;
            const int kc = k;
            k += LPE;
            item = k < nOrd ? ent(k) : IT_NONE;
            if ((cur & IT_GEN) != 0u) solveVelocityGeneralNI(*this, genSlot(kc));
            else solveVelocitySimple(kc, cur);
          }
          g.usync();
        }
      }
      if (c0) rec4(2 * g.lane).set(3, q0.w);   // the accumulated impulse, for storeSimple
    }
    KB_T(5);
#pragma unroll 1
    for (int e = g.lane; e < nOrd; e += LPE) {
      if ((ent(e) & IT_GEN) != 0u) storeGeneralNI(*this, genSlot(e));
      else storeSimple(e, (int)entC(e), ent(e));
    }
    // ---- integrate positions
#pragma unroll 1
    for (int b = g.lane; b < B; b += LPE) {
      if (isl(b) < 0) continue;
      float4 p = pos4(b);
      float4 v = vel4(b);
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
      pos4(b) = p;
      vel4(b) = v;
    }
    g.usync();
    KB_T(6);
    // ---- position iterations with per-island early exit (b2Island::Solve breaks out of the loop of an island as
    //      soon as one sweep leaves every separation above -3 linearSlop).  `unsolved` (one bit per island,
    //      identical in every lane) is the set of islands still iterating.
    {
      unsigned long long unsolved = nIslands >= 64 ? ~0ull : ((1ull << nIslands) - 1ull);
      for (int it = 0; it < L.posIters; ++it) {
        if (!g.uany(unsolved != 0ull)) break;
        nPit += (uint32_t)__popcll(unsolved);
        unsigned long long bad = 0ull;  // islands with a constraint of this lane below the limit in this sweep
        int k = g.lane;
        uint32_t item = k < nOrd ? ent(k) : IT_NONE;
        for (int r = 0; r < nRowsU; ++r) {
          if (IT_ROW(item) == r) {
            const uint32_t cur = item;
            const int kc = k;
            k += LPE;
            item = k < nOrd ? ent(k) : IT_NONE;
            const int island = IT_ISL(cur);
            if (((unsolved >> island) & 1ull) != 0ull) {
              const bool ok = (cur & IT_FAST) != 0u ? solvePositionFast(kc, cur)
                              : ((cur & IT_GEN) != 0u ? solvePositionGeneralNI(*this, genSlot(kc))
                                                      : solvePositionSimple(kc, cur));
              if (!ok) bad |= 1ull << island;
            }
          }
          g.usync();
        }
        // (the sweep loop is warp-uniform; envs of one batch share B, so `nIslands >= 32` could only differ between
        //  groups in its value, never in whether the second word exists)
        unsigned long long badAll = (unsigned long long)g.ured_or((uint32_t)bad);
        if (L.B > 32) badAll |= (unsigned long long)g.ured_or((uint32_t)(bad >> 32)) << 32;
        unsolved &= badAll;
      }
      // bit 1: positionSolved (sleep bookkeeping below adds bit 2: minSleepTime < timeToSleep)
#pragma unroll 1
      for (int i = g.lane; i < nIslands; i += LPE) islflag(i) = ((unsolved >> i) & 1ull) != 0ull ? 0u : 2u;
      g.usync();
    }
    KB_T(7);
    // ---- copy back: SynchronizeTransform; sleep bookkeeping
#pragma unroll 1
    for (int b = g.lane; b < B; b += LPE) {
      const int island = isl(b);
      if (island < 0) continue;
      const float4 p = pos4(b);
      const float4 k = bc4(b);
      Rot q = rot_set(p.z);
      V2 o = mk(p.x, p.y) - rmul(q, mk(k.z, k.w));
      xf4(b) = make_float4(o.x, o.y, q.s, q.c);
      if (L.enableSleep) {
        const float4 v = vel4(b);
        const float linTolSqr = KB_LIN_SLEEP_TOL * KB_LIN_SLEEP_TOL;
        const float angTolSqr = KB_ANG_SLEEP_TOL * KB_ANG_SLEEP_TOL;
        float st;
        if (v.z * v.z > angTolSqr || dot(mk(v.x, v.y), mk(v.x, v.y)) > linTolSqr) {
          st = 0.0f;
        } else {
          st = p.w + h;
        }
        pos4(b).set(3, st);
        if (!(st >= KB_TIME_TO_SLEEP)) islflag(island).atomOr(4u);  // minSleepTime < timeToSleep
      }
    }
    g.usync();
    if (L.enableSleep) {
#pragma unroll 1
      for (int b = g.lane; b < B; b += LPE) {
        const int island = isl(b);
        if (island < 0) continue;
        const uint32_t f = islflag(island);
        if ((f & 4u) == 0u && (f & 2u) != 0u) {
          // b2Body::SetAwake(false)
          vel4(b) = make_float4(0.0f, 0.0f, 0.0f, u2f(f2u(vel4(b).get(3)) & ~BF_AWAKE));
          pos4(b).set(3, 0.0f);
        }
      }
      g.usync();
    }
    g.usync();
    KB_T(8);
    synchronizeFixtures(false);
    KB_T(9);
    findNewContactsT<true>();   // u-variants degrade to the group's own outside uniform mode (reset kernel)
    g.usync();
    KB_T(10);
  }

  // shape AABB of proxy p under transform xf (b2Shape::ComputeAABB)
  __device__ __forceinline__ void shapeAABB(int p, Xf xf, V2* lo, V2* hi) {
    const ProxyConst* pc = px + p;
    const int type = ptype(p);
    if (type == SHAPE_CIRCLE) {
      const float r = pradius(p);
      V2 c = xf.p + rmul(xf.q, mk(0.0f, 0.0f));
      *lo = mk(c.x - r, c.y - r);
      *hi = mk(c.x + r, c.y + r);
    } else if (type == SHAPE_POLYGON) {
      const int n = __ldg(&pc->count);
      V2 lower = xmul(xf, pvert(pc, 0));
      V2 upper = lower;
      for (int i = 1; i < n; ++i) {
        V2 v = xmul(xf, pvert(pc, i));
        lower = mk(b2min(lower.x, v.x), b2min(lower.y, v.y));
        upper = mk(b2max(upper.x, v.x), b2max(upper.y, v.y));
      }
      const float r = __ldg(&pc->radius);
      *lo = mk(lower.x - r, lower.y - r);
      *hi = mk(upper.x + r, upper.y + r);
    } else {
      V2 a = xmul(xf, pvert(pc, 1));
      V2 b = xmul(xf, pvert(pc, 2));
      *lo = mk(b2min(a.x, b.x), b2min(a.y, b.y));
      *hi = mk(b2max(a.x, b.x), b2max(a.y, b.y));
    }
  }

  // b2Body::SynchronizeFixtures + b2BroadPhase::MoveProxy for every body that was in an island
  // (toiMode: for bodies flagged in isl() by the TOI mini-island; xf1 is rebuilt from (c0, a0)).
  __device__ __forceinline__ void synchronizeFixtures(bool toiMode) {
    uint32_t mlo = 0u, mhi = 0u;
#pragma unroll 1
    for (int p = g.lane; p < L.P; p += LPE) {
      const int b = pbody(p);
      if (b == S) continue;
      if (isl(b) < 0) continue;
      const float4 sw = sweep4(b);
      const float4 k = bc4(b);
      Xf xf1;
      if (toiMode) {
        xf1.q = rot_set(sw.z);
      } else {
        const float2 oq = oldq(b);
        xf1.q.s = oq.x;
        xf1.q.c = oq.y;
      }
      xf1.p = mk(sw.x, sw.y) - rmul(xf1.q, mk(k.z, k.w));
      const Xf xf2 = bodyXf(b);
      V2 lo1, hi1, lo2, hi2;
      shapeAABB(p, xf1, &lo1, &hi1);
      shapeAABB(p, xf2, &lo2, &hi2);
      const V2 lo = mk(b2min(lo1.x, lo2.x), b2min(lo1.y, lo2.y));
      const V2 hi = mk(b2max(hi1.x, hi2.x), b2max(hi1.y, hi2.y));
      const V2 displacement = xf2.p - xf1.p;
      const float4 fat = fat4(p);
      const bool contains = fat.x <= lo.x && fat.y <= lo.y && hi.x <= fat.z && hi.y <= fat.w;
      if (!contains) {
        float4 nb = make_float4(lo.x - KB_AABB_EXTENSION, lo.y - KB_AABB_EXTENSION, hi.x + KB_AABB_EXTENSION,
                                hi.y + KB_AABB_EXTENSION);
        const V2 d = KB_AABB_MULTIPLIER * displacement;
        if (d.x < 0.0f) nb.x += d.x; else nb.z += d.x;
        if (d.y < 0.0f) nb.y += d.y; else nb.w += d.y;
        fat4(p) = nb;
        if (p < 32) mlo |= 1u << p; else mhi |= 1u << (p - 32);
      }
    }
    // (from solve() this is warp-uniform control flow; the TOI caller is not)
    mlo = toiMode ? g.red_or(mlo) : g.ured_or(mlo);
    if (L.P > 32) mhi = toiMode ? g.red_or(mhi) : g.ured_or(mhi);
    if (g.lane == 0) {
      hdr(H_MOVED) |= mlo;
      if (L.P > 32) hdr(H_MOVED + 1) |= mhi;
    }
    if (toiMode) g.sync(); else g.usync();
  }

  // b2BroadPhase::UpdatePairs + b2ContactManager::AddPair.  Pairs (i < j) with a moved member are
  // created in (i, j) order == Box2D's sorted pair buffer, so creation order matches.  A lane owns a
  // row i: it tests the columns j > i that need testing (row or column moved, no contact yet) and
  // collects the new pairs in a 64-bit mask; an exclusive scan over the rows of a chunk gives every
  // row its place in the contact list.  Rows are independent: a new pair (i, j) never changes what a
  // later row has to test.
  // U: called from warp-uniform control flow (solve() in uniform mode): the loops run the warp's maximal trip counts,
  // groups without work run them empty, and the votes / scans are the full-mask forms.  The TOI path and the reset
  // kernel call the group form.
  __device__ __forceinline__ void findNewContacts() { findNewContactsT<false>(); }
  template <bool U>
  __device__ __forceinline__ void findNewContactsT() {
    const uint32_t mlo = hdr(H_MOVED), mhi = hdr(H_MOVED + 1);
    if (U) g.usync(); else g.sync();
    const bool some = (mlo | mhi) != 0u;
    if (U ? !g.uany(some) : !some) return;
    if (some && g.lane == 0) {
      hdr(H_MOVED) = 0u;
      hdr(H_MOVED + 1) = 0u;
    }
    const int P = L.P;
    const unsigned long long valid = P >= 64 ? ~0ull : ((1ull << P) - 1ull);
    const unsigned long long moved = ((unsigned long long)mlo | ((unsigned long long)mhi << 32)) & valid;
    int nC = (int)hdr(H_NC);
    bool overflow = false;
    uint32_t tests = 0u;
#pragma unroll 1
    for (int ib = 0; ib < P - 1; ib += LPE) {
      const bool more = (moved >> ib) != 0ull;   // a row from here on, or one of their columns, moved
      if (U ? !g.uany(more) : !more) break;
      const int i = ib + g.lane;
      unsigned long long cand = 0ull;
      int bi = S;
      if (i < P - 1) {
        const bool movedI = ((moved >> i) & 1ull) != 0ull;
        unsigned long long cols = (movedI ? valid : moved) & (~0ull << (i + 1));
        if (cols != 0ull) {
          tests += (uint32_t)__popcll(cols);
          cols &= ~((unsigned long long)(uint32_t)adj(i, 0) | ((unsigned long long)(uint32_t)adj(i, 1) << 32));
          if (cols != 0ull) {
            const float4 fi = fat4(i);
            bi = pbody(i);
            while (cols != 0ull) {
              const int j = __ffsll((long long)cols) - 1;
              cols &= cols - 1ull;
              const float4 fj = fat4(j);
              // b2TestOverlap
              const bool overlap = !(fj.x - fi.z > 0.0f || fj.y - fi.w > 0.0f || fi.x - fj.z > 0.0f || fi.y - fj.w > 0.0f);
              if (overlap && pbody(j) != bi) cand |= 1ull << j;
            }
          }
        }
      }
      const int cnt = __popcll(cand);
      const uint32_t newMask = U ? g.uballot(cnt != 0) : g.ballot(cnt != 0);
      if (U ? !g.uany(newMask != 0u) : newMask == 0u) continue;
      const int off = U ? g.uexscan(cnt) : g.exscan(cnt);
      const int total = U ? g.ubcast(off + cnt, LPE - 1) : g.bcast(off + cnt, LPE - 1);
      if (cnt != 0) {
        int dst = nC + off;
        const int ti = ptype(i);
        const int rankI = ti == SHAPE_EDGE ? 0 : (ti == SHAPE_POLYGON ? 1 : 2);
        wake(bi);
        while (cand != 0ull) {
          const int j = __ffsll((long long)cand) - 1;
          cand &= cand - 1ull;
          if (dst < L.Cmax) {
            // type register: chain edge < polygon < circle takes the A slot (b2Contact::Create)
            const int tj = ptype(j);
            const int rankJ = tj == SHAPE_EDGE ? 0 : (tj == SHAPE_POLYGON ? 1 : 2);
            const int pa = rankI > rankJ ? j : i, pb = rankI > rankJ ? i : j;
            cw(dst) = (uint32_t)pa | ((uint32_t)pb << 8) | CI_ENABLED;
            adj(i, j >> 5).atomOr(1u << (j & 31));
            adj(j, i >> 5).atomOr(1u << (i & 31));
            wake(pbody(j));
          } else {
            overflow = true;
          }
          ++dst;
        }
      }
      nC = min(nC + total, L.Cmax);
    }
    nTests += U ? g.ured_add(tests) : g.red_add(tests);
    const uint32_t ovMask = U ? g.uballot(overflow) : g.ballot(overflow);
    if (some && g.lane == 0) {
      hdr(H_NC) = (uint32_t)nC;
      if (ovMask != 0u) hdr(H_STATUS) |= KB_STATUS_CONTACT_OVERFLOW;
    }
    if (U) g.usync(); else g.sync();
  }

  // b2World::Step(dt, velIters, posIters)
  __device__ __forceinline__ void worldStep() {
    nSub += 1u;
    nCon += hdr(H_NC);
    KB_T(0);
    collide();
    g.usync();
    KB_T(1);
    solve();
    if (L.enableToi) {
      // any contact with the table at all?  (the common case is none: skip the out-of-line TOI path)
      const int nC = (int)hdr(H_NC);
      bool wallContact = false;
#pragma unroll 1
      for (int i = g.lane; i < nC; i += LPE) wallContact |= pbody(CW_PA(cw(i))) == S;
      const uint32_t wallMask = g.uballot(wallContact);
      if (wallMask != 0u) nToi += solveTOINI(*this);
      g.usync();
      KB_T(11);
    }
  }

  __device__ __forceinline__ void solveTOI();   // kb_toi.cuh

  // ----------------------------------------------------------------------------- outputs
  // get_state (kilobots_env.py:115-118) + the reward / done / info hooks (:123-131)
  __device__ __forceinline__ void gather(const KernelArgs& a, int env) {
    g.sync();   // padding groups skip gather: not warp-uniform
    const int M = L.M, N = L.N;
    bool bad = false;
    float* flat = a.obsFlat ? a.obsFlat + (size_t)env * (2 * N + L.L + 4 * M) : nullptr;
#pragma unroll 1
    for (int b = g.lane; b < L.B; b += LPE) {
      float4 x = xf4(b);
      float ang = pos4(b).get(2);
      float ox = (float)((double)x.x / 25.0), oy = (float)((double)x.y / 25.0);
      if (bkind(b) == KB_BODY_ABSENT) {   // an absent body's rows are quiet NaN: never read as a body at the origin
        ox = oy = ang = x.z = x.w = __int_as_float(0x7FC00000);
      } else {
        bad |= !(isfinite(x.x) && isfinite(x.y) && isfinite(ang));
      }
      float* o = b < M ? (a.obsObjects ? a.obsObjects + ((size_t)env * M + b) * 3 : nullptr)
                       : (a.obsKilobots ? a.obsKilobots + ((size_t)env * N + (b - M)) * 3 : nullptr);
      if (o) {
        o[0] = ox;
        o[1] = oy;
        o[2] = ang;
      }
      if (flat) {
        // YamlKilobotsEnv.observation_space layout (yaml_kilobots_env.py:163-178)
        if (b < M) {
          float* f = flat + 2 * N + L.L + 4 * b;
          f[0] = ox; f[1] = oy; f[2] = x.z; f[3] = x.w;   // xf.q = (sin, cos) of the body angle
        } else {
          flat[2 * (b - M)] = ox;
          flat[2 * (b - M) + 1] = oy;
        }
      }
    }
    if (g.any(bad) && g.lane == 0) hdr(H_STATUS) |= KB_STATUS_NONFINITE;
    observeLights(*this, a, env, flat, g.lane, LPE);
    g.sync();   // padding groups skip gather: not warp-uniform
    if (g.lane == 0) taskEnd(*this, a, env);
  }
};

template <int LPE, bool UNI, class LT>
__device__ __noinline__ void warmStartGeneralNI(Sim<LPE, UNI, LT> s, int q) { s.warmStartGeneral(q); }
template <int LPE, bool UNI, class LT>
__device__ __noinline__ void solveVelocityGeneralNI(Sim<LPE, UNI, LT> s, int q) { s.solveVelocityGeneral(q); }
template <int LPE, bool UNI, class LT>
__device__ __noinline__ bool solvePositionGeneralNI(Sim<LPE, UNI, LT> s, int q) {
  return s.solvePositionGeneral(q, KB_BAUMGARTE, -3.0f * KB_LINEAR_SLOP, -1, -1);
}
template <int LPE, bool UNI, class LT>
__device__ __noinline__ void initGeneralNI(Sim<LPE, UNI, LT> s, int q, int ci, uint32_t item) {
  s.initGeneral(q, ci, IT_BA(item), IT_BB(item), (uint32_t)ci | ((uint32_t)IT_ISL(item) << 16), false);
}
template <int LPE, bool UNI, class LT>
__device__ __noinline__ void storeGeneralNI(Sim<LPE, UNI, LT> s, int q) { s.storeGeneral(q); }

}  // namespace kb
