// kb_swarm.cuh -- the large-swarm tier: ONE CTA per environment, up to 2040 kilobots (proxy ids are 11 bits wide; the
// shared-memory image is ~35 bytes per body + ~21 per touching contact of capacity).
//
// BASELINE.json configs[3] ("256 envs x 1024 kilobots, grid broadphase, dense contacts"): the reference puts no
// bound on kilobots per env (gym_kilobots/envs/kilobots_env.py:105-109, yaml_kilobots_env.py:327-354 kilobots.num),
// and the lane-group kernel of kb_step.cuh stops at 62 bodies (64-bit adjacency masks).  Same semantics, same
// Box2D orderings, different data structures:
//   * body state (c, a, sleepTime | v, w, flags) stays in shared memory for all sub-steps of an action; fat AABBs,
//     the persistent contact list (flags word + proxy-pair word + 8-word manifold record per contact), controller
//     state, sweeps, (sin, cos), the level schedule, the solver's records and the pair hash live in the env's
//     L2-resident blob and are streamed by the data-parallel phases / prefetched by the relay's waiting warps;
//   * broadphase = per-env UNIFORM GRID over the fat-AABB centres of the dynamic proxies (counting sort; the
//     per-cell counts are accumulated with warp-aggregated atomics: __match_any_sync groups the lanes that hit the
//     same cell, the leader adds the group's popcount and the ranks come from the lane mask).  Every proxy owns
//     the candidate pairs (i, j > i) it finds in the 3x3 (or wider, if some proxy is large) neighbourhood of its
//     cell, an open-addressing hash of the existing pairs stands in for b2ContactManager::AddPair's list walk, and
//     a block-wide exclusive scan over the per-proxy counts places the new pairs in (proxyA, proxyB)-sorted order
//     -- exactly the order b2BroadPhase::UpdatePairs hands them to AddPair, so contact creation order matches;
//   * islands: per-body CSR lists over the touching list (descending contact index == Box2D's LIFO contact-edge
//     lists), DFS in Box2D's order on warp 0 (a body's contact edges side by side on the lanes), dependency level
//     per constraint, counting sort by level, wide levels cut into rows of at most 8;
//   * solver: the constraints of one level touch disjoint bodies, so a sweep over levels is bit-identical to
//     Box2D's sequential sweep.  A lattice swarm is ONE island whose level structure is a long chain (1-3
//     constraints per level): the rows are executed as a RELAY over the CTA's warps -- four rows per turn in lane
//     groups of eight, the turn's entries and records (3 x float4 per constraint) fetched from L2 while the seven
//     turns before it run, hand-over on named barriers (see "relay" below and DESIGN.md section 6).
// Scope of this tier (checked by kb_create): every dynamic body is a kilobot (one circle fixture at the body origin,
// friction 0, restitution 0), no pushable objects (M = 0); the table's chain edges are the only other proxies.
// All constraints are therefore "simple" (one manifold point, frictionless, no restitution): kb_step.cuh's
// initSimple / warmStartSimple / solveVelocitySimple / solvePositionSimple arithmetic, restated here on the swarm
// layout; continuous collision (b2World::SolveTOI) is the table-edge-against-circle case of kb_toi.cuh.
#pragma once
#include "kb_toi.cuh"

namespace kb {

// threads per CTA: 512, 256 or 128 -- the widest block that still lets as many CTAs share an SM as its shared memory holds
// (<= 128 registers per thread: 512 threads x 1 CTA, 256 x 2, 128 x 4).  A second CTA on the SM overlaps with the first
// (the solver's dependent chain keeps one warp at a time busy): 296 envs of 484 kilobots take as long as 148.
#define KB_SWARM_THREADS_MAX 512
#define KB_SWARM_MAX_BODIES 2040   /* 11-bit proxy ids (bodies + table edges < 2048) */

// swarm manifold record (8 words per contact, HBM/L2)
#define SR_LNX 0
#define SR_LNY 1
#define SR_LPX 2
#define SR_LPY 3
#define SR_IMP 4    /* normal impulse of the one manifold point (warm start) */
#define SR_ID 5     /* b2ContactID key of the point */
#define SR_TYPE 6   /* manifold type | pointCount << 8 */
#define SR_WORDS 8

#define SW_NOISLAND 0xFFFFu
#define SW_LONELY 0xFFFEu   /* awake body without touching contacts: an island of its own */

// phase timers (only with -DKB_PROFILE; compiled out of the product library): cycles of thread 0 between marks
#ifdef KB_PROFILE
#define SW_T(i)                          \
  do {                                   \
    __syncthreads();                     \
    const long long now_ = clock64();    \
    tp[i] += now_ - tlast;               \
    tlast = now_;                        \
  } while (0)
#else
#define SW_T(i) do { } while (0)
#endif

// proxies standing in for references into the env's blob (HBM / L2)
struct GF2 {
  float2* p;
  __device__ __forceinline__ operator float2() const { return *p; }
  __device__ __forceinline__ void operator=(float2 v) const { *p = v; }
};
struct GF4 {
  float4* p;
  __device__ __forceinline__ operator float4() const { return *p; }
  __device__ __forceinline__ void operator=(float4 v) const { *p = v; }
  __device__ __forceinline__ float get(int i) const { return reinterpret_cast<const float*>(p)[i]; }
  __device__ __forceinline__ void set(int i, float v) const { reinterpret_cast<float*>(p)[i] = v; }
};
struct GU32 {
  uint32_t* p;
  __device__ __forceinline__ operator uint32_t() const { return *p; }
  __device__ __forceinline__ uint32_t operator=(uint32_t v) const { *p = v; return v; }
};
struct GU16 {
  uint16_t* p;
  __device__ __forceinline__ operator uint32_t() const { return (uint32_t)*p; }
  __device__ __forceinline__ void operator=(uint32_t v) const { *p = (uint16_t)v; }
};

template <int NT>
struct Swarm {
  const Layout& L;
  const SwarmLayout& W;
  uint32_t sa;          // shared-window byte address of the CTA's dynamic shared memory
  float* blob;
  const ProxyConst* px;
  const BodyConst* bc;
  int tid, S, nWall;
  int nP;               // the scene's proxies: nWall + its kilobots (absent bodies own none); L.P is the batch's maximum
  uint32_t nSub, nCon, nPts, nLvl, nPit, nToi, nTests, nIsl;   // thread 0's copy is flushed
#ifdef KB_PROFILE
  long long tp[KB_PROF_SLOTS], tlast;
#endif

  __device__ __forceinline__ Swarm(const Layout& l, const SwarmLayout& w) : L(l), W(w) {
    nSub = nCon = nPts = nLvl = nPit = nToi = nTests = nIsl = 0u;
#ifdef KB_PROFILE
    for (int i = 0; i < KB_PROF_SLOTS; ++i) tp[i] = 0;
    tlast = clock64();
#endif
    sa = (uint32_t)__cvta_generic_to_shared(kb_smem);
    tid = threadIdx.x;
    S = l.B;
  }
  // ---- shared memory (byte offsets from W)
  __device__ __forceinline__ SF4 pos4(int b) const { return SF4{sa + W.zPos + 16u * (uint32_t)b}; }   // cx cy a sleepTime
  __device__ __forceinline__ SF4 vel4(int b) const { return SF4{sa + W.zVel + 16u * (uint32_t)b}; }   // vx vy w flags
  // (sin, cos) of the body angle: the q half of the blob's xf4 rows (the static slot B holds (0, 1))
  __device__ __forceinline__ GF2 q2(int b) const { return GF2{reinterpret_cast<float2*>(blob + L.oXf + 4 * b + 2)}; }
  __device__ __forceinline__ float2 massOf(int b) const { return make_float2(__ldg(&bc[b].invMass), __ldg(&bc[b].invI)); }
  __device__ __forceinline__ int bkind(int b) const { return __ldg(&bc[b].kind); }
  __device__ __forceinline__ SF4 dummy4() const { return SF4{sa + W.zDummy + 16u * (uint32_t)(tid & 31)}; }
  __device__ __forceinline__ SU32 hdr(int i) const { return SU32{sa + W.zHdr + 4u * (uint32_t)i}; }
  __device__ __forceinline__ SU32 moved(int w) const { return SU32{sa + W.zMoved + 4u * (uint32_t)w}; }
  __device__ __forceinline__ SU32 misc(int i) const { return SU32{sa + W.zMisc + 4u * (uint32_t)i}; }
  __device__ __forceinline__ SU16 isl(int b) const { return SU16{sa + W.zIsl + 2u * (uint32_t)b}; }
  __device__ __forceinline__ uint32_t islStateAddr(int i) const { return sa + W.zIslState + (uint32_t)i; }
  // the level schedule and the solver's records live in the blob (L2-resident, fetched by the relay's waiting warps): that
  // keeps the CTA's shared memory small enough for TWO CTAs per SM at 1024 kilobots, and a second CTA overlaps perfectly
  __device__ __forceinline__ GU32 ent0(int e) const { return GU32{reinterpret_cast<uint32_t*>(blob + W.oEnt0) + e}; }        // bA | bB << 16
  __device__ __forceinline__ GU16 entC(int e) const { return GU16{reinterpret_cast<uint16_t*>(blob + W.oEntC) + e}; }        // contact index
  __device__ __forceinline__ GU16 entI(int e) const { return GU16{reinterpret_cast<uint16_t*>(blob + W.oEntI) + e}; }        // island | fast << 15
  __device__ __forceinline__ GU16 rowStart(int l) const { return GU16{reinterpret_cast<uint16_t*>(blob + W.oRow) + l}; }
  // three float4 per schedule entry: two phase-dependent records and the masses (invMassA, invIA, invMassB, invIB)
  __device__ __forceinline__ GF4 rec4(int i) const { return GF4{reinterpret_cast<float4*>(blob + W.oRec) + i}; }
  __device__ __forceinline__ uint16_t* tlCp() const { return reinterpret_cast<uint16_t*>(blob + W.oTlC); }
  __device__ __forceinline__ uint32_t* hashp() const { return reinterpret_cast<uint32_t*>(blob + W.oHash); }
  __device__ __forceinline__ SF64Arr lightState() const { return SF64Arr{sa + W.zLight}; }
  __device__ __forceinline__ LCs lightConst(int l) const { return LCs{sa + W.zLc + 4u * LC_WORDS * (uint32_t)l}; }
  // scratch views (alias the record region; each is live only inside the phase that names it)
  __device__ __forceinline__ uint32_t scr(int off) const { return sa + W.zScr + (uint32_t)off; }
  // ---- blob (HBM / L2)
  __device__ __forceinline__ float4* fatp() const { return reinterpret_cast<float4*>(blob + L.oFat); }
  __device__ __forceinline__ uint32_t* cwp() const { return reinterpret_cast<uint32_t*>(blob + L.oCw); }
  __device__ __forceinline__ uint32_t* cpairp() const { return reinterpret_cast<uint32_t*>(blob + W.oCpair); }
  __device__ __forceinline__ float* recp(int i) const { return blob + L.oMan + SR_WORDS * i; }
  __device__ __forceinline__ float4* sweepp() const { return reinterpret_cast<float4*>(blob + W.oSweep); }   // c0x c0y a0 alpha0
  __device__ __forceinline__ float* toip() const { return blob + L.oToi; }
  __device__ __forceinline__ double* ctrl(int k) const { return reinterpret_cast<double*>(blob + L.oCtrl) + 4 * k; }

  __device__ __forceinline__ int pbody(int p) const { return p < nWall ? S : p - nWall; }
  __device__ __forceinline__ Xf bodyXf(int b) const {
    const float4 p = pos4(b);
    const float2 q = q2(b);
    Xf t;
    t.p = mk(p.x, p.y);   // local centre is zero for every body of this tier: xf.p == c
    t.q.s = q.x;
    t.q.c = q.y;
    return t;
  }
  // the position the task and the observations read: c (== xf.p), from shared memory
  __device__ __forceinline__ float2 obsPos(int b) const {
    const float4 p = pos4(b);
    return make_float2(p.x, p.y);
  }
  __device__ __forceinline__ bool awake(int b) const { return (f2u(vel4(b).get(3)) & BF_AWAKE) != 0u; }
  __device__ __forceinline__ void wake(int b) const {
    if (b == S) return;
    const uint32_t f = f2u(vel4(b).get(3));
    if ((f & BF_AWAKE) == 0u) {
      vel4(b).set(3, u2f(f | BF_AWAKE));
      pos4(b).set(3, 0.0f);
    }
  }

  // ---- block-wide primitives (every thread of the CTA calls them)
  // exclusive prefix sum of v over the threads; *total = sum.  Uses misc words 16..48.
  __device__ __forceinline__ int blockExScan(int v, int* total) const {
    const int lane = tid & 31, wid = tid >> 5;
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xFFFFFFFFu, x, d);
      if (lane >= d) x += y;
    }
    __syncthreads();   // previous users of the warp-sum words are done
    if (lane == 31) misc(16 + wid) = (uint32_t)x;
    __syncthreads();
    const int nw = NT / 32;
    int ws = lane < nw ? (int)misc(16 + lane) : 0;
    int wx = ws;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xFFFFFFFFu, wx, d);
      if (lane >= d) wx += y;
    }
    const int woff = __shfl_sync(0xFFFFFFFFu, wx - ws, wid);
    *total = __shfl_sync(0xFFFFFFFFu, wx, nw - 1);
    return woff + x - v;
  }

  // ------------------------------------------------------------------------- state I/O
  __device__ __forceinline__ void loadState() {
    const float4* bp = reinterpret_cast<const float4*>(blob + L.oPos);
    const float4* bv = reinterpret_cast<const float4*>(blob + L.oVel);
#pragma unroll 1
    for (int b = tid; b <= L.B; b += NT) {
      if (b < L.B) {
        pos4(b) = bp[b];
        vel4(b) = bv[b];
      } else {
        pos4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        vel4(b) = make_float4(0.0f, 0.0f, 0.0f, u2f(BF_AWAKE));
        q2(b) = make_float2(0.0f, 1.0f);
      }
    }
    const uint32_t* bw = reinterpret_cast<const uint32_t*>(blob);
    for (int i = tid; i < H_WORDS; i += NT) hdr(i) = bw[L.oHdr + i];
    for (int i = tid; i < W.movedWords; i += NT) moved(i) = bw[W.oMoved + i];
    for (int i = tid; i < 2 * L.L; i += NT) sts_u32(sa + W.zLight + 4u * (uint32_t)i, bw[L.oLight + i]);
    __syncthreads();
  }
  __device__ __forceinline__ void loadConsts(const LightConst* lights) {
    for (int w = tid; w < LC_WORDS * L.numLights; w += NT)
      sts_u32(sa + W.zLc + 4u * (uint32_t)w, __ldg(reinterpret_cast<const uint32_t*>(lights) + w));
    __syncthreads();
  }
  __device__ __forceinline__ void storeState() {
    __syncthreads();
    float4* bp = reinterpret_cast<float4*>(blob + L.oPos);
    float4* bv = reinterpret_cast<float4*>(blob + L.oVel);
    float4* bx = reinterpret_cast<float4*>(blob + L.oXf);
#pragma unroll 1
    for (int b = tid; b < L.B; b += NT) {
      const float4 p = pos4(b);
      bp[b] = p;
      bv[b] = vel4(b);
      reinterpret_cast<float2*>(bx + b)[0] = make_float2(p.x, p.y);   // xf.p == c (zero local centres); xf.q is kept in place
    }
    uint32_t* bw = reinterpret_cast<uint32_t*>(blob);
    for (int i = tid; i < H_WORDS; i += NT) bw[L.oHdr + i] = hdr(i);
    for (int i = tid; i < W.movedWords; i += NT) bw[W.oMoved + i] = moved(i);
    for (int i = tid; i < 2 * L.L; i += NT) bw[L.oLight + i] = lds_u32(sa + W.zLight + 4u * (uint32_t)i);
    if (tid == 0) {
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

  // --------------------------------------------------------------------------- collide
  // b2Contact::Update for contact i (this thread).  Returns true if touching changed.
  __device__ __forceinline__ bool updateContact(int i) const {
    uint32_t w = cwp()[i];
    const uint32_t pr = cpairp()[i];
    const int pa = (int)(pr & 0xFFFFu), pb = (int)(pr >> 16);
    const int bA = pbody(pa), bB = pbody(pb);
    const int oldPC = (w & CI_PC_MASK) >> CI_PC_SHIFT;
    const bool wasTouching = (w & CI_TOUCHING) != 0u;
    Manifold m;
    m.pointCount = 0;
    m.type = 0;
    m.lnx = m.lny = m.lpx = m.lpy = 0.0f;
    m.px[0] = m.py[0] = m.px[1] = m.py[1] = 0.0f;
    m.id[0] = m.id[1] = 0u;
    const float rB = __ldg(&px[pb].radius);
    if (pa >= nWall) collide_circles(m, __ldg(&px[pa].radius), bodyXf(bA), rB, bodyXf(bB));
    else collide_edge_circle(m, px + pa, bodyXf(bA), rB, bodyXf(bB));
    const bool touching = m.pointCount > 0;
    if (touching) {
      float4* rec = reinterpret_cast<float4*>(recp(i));
      float ni = 0.0f;
      if (oldPC > 0) {
        const float4 r1 = rec[1];   // imp id type pad
        if (f2u(r1.y) == m.id[0]) ni = r1.x;
      }
      rec[0] = make_float4(m.lnx, m.lny, m.lpx, m.lpy);
      rec[1] = make_float4(ni, u2f(m.id[0]), u2f((uint32_t)m.type | (1u << 8)), 0.0f);
    }
    w |= CI_ENABLED;
    w = touching ? (w | CI_TOUCHING) : (w & ~CI_TOUCHING);
    w = (w & ~CI_PC_MASK) | ((uint32_t)m.pointCount << CI_PC_SHIFT);
    cwp()[i] = w;
    return touching != wasTouching;
  }

  // b2ContactManager::Collide.  World-list order is descending array index; a sleeping pair is only visited if an
  // earlier (higher index) contact woke one of its bodies: wakeAt[b] = highest contact index that woke b
  // (fix-point over passes; a pass visits every not-yet-visited contact that is eligible under the current wakeAt).
  __device__ __forceinline__ void collide() {
    const int nC = (int)hdr(H_NC);
    if (nC == 0) return;
    bool sleepy = false;
#pragma unroll 1
    for (int b = tid; b < L.B; b += NT) sleepy |= !awake(b);
    const bool anyAsleep = __syncthreads_or(sleepy) != 0;
    const uint32_t wakeAt = scr(W.cWakeAt);
    if (anyAsleep) {
#pragma unroll 1
      for (int b = tid; b <= L.B; b += NT) sts_u32(wakeAt + 4u * (uint32_t)b, awake(b) && b != S ? 0x7FFFFFFFu : 0xFFFFFFFFu);
      __syncthreads();
    }
    bool anyDestroyed = false;
    for (int pass = 0;; ++pass) {
      bool woke = false;
#pragma unroll 1
      for (int i = tid; i < nC; i += NT) {
        uint32_t w = cwp()[i];
        if ((w & CI_DONE) != 0u) continue;
        const uint32_t pr = cpairp()[i];
        const int pa = (int)(pr & 0xFFFFu), pb = (int)(pr >> 16);
        const int bA = pbody(pa), bB = pbody(pb);
        if (anyAsleep) {
          const bool actA = bA != S && (int32_t)lds_u32(wakeAt + 4u * (uint32_t)bA) > i;
          const bool actB = bB != S && (int32_t)lds_u32(wakeAt + 4u * (uint32_t)bB) > i;
          if (!(actA || actB)) continue;
        }
        const float4 fa = fatp()[pa], fb = fatp()[pb];
        const bool overlap = !(fb.x - fa.z > 0.0f || fb.y - fa.w > 0.0f || fa.x - fb.z > 0.0f || fa.y - fb.w > 0.0f);
        bool wakeEvent;
        if (!overlap) {
          wakeEvent = (w & CI_PC_MASK) != 0u;
          cwp()[i] = w | CI_DESTROY | CI_DONE;
          anyDestroyed = true;
        } else {
          wakeEvent = updateContact(i);
          if (anyAsleep) cwp()[i] |= CI_DONE;
        }
        if (wakeEvent && anyAsleep) {
          if (bA != S) SI32{wakeAt + 4u * (uint32_t)bA}.atomMax(i);
          if (bB != S) SI32{wakeAt + 4u * (uint32_t)bB}.atomMax(i);
          woke = true;
        }
      }
      if (!anyAsleep) break;
      if (__syncthreads_or(woke) == 0) break;
    }
    __syncthreads();
    if (anyAsleep) {
#pragma unroll 1
      for (int b = tid; b < L.B; b += NT)
        if ((int32_t)lds_u32(wakeAt + 4u * (uint32_t)b) >= 0) wake(b);
    }
    const bool compact = __syncthreads_or(anyDestroyed) != 0;
    if (!compact && !anyAsleep) return;
    // clear DONE marks; stable compaction (chunks of the CTA's width: all reads of a chunk precede its writes, and
    // a chunk only writes at or below its own first index)
    int out = 0;
#pragma unroll 1
    for (int base = 0; base < nC; base += NT) {
      const int i = base + tid;
      uint32_t w = 0u, pr = 0u;
      bool keep = false;
      if (i < nC) {
        w = cwp()[i];
        pr = cpairp()[i];
        keep = (w & CI_DESTROY) == 0u;
        w &= ~(CI_DONE | CI_DESTROY);
      }
      if (!compact) {
        if (i < nC) cwp()[i] = w;
        continue;
      }
      int total;
      const int dst = out + blockExScan(keep ? 1 : 0, &total);
      float4 r0, r1;
      float toi = 0.0f;
      const bool moveRec = keep && dst != i;
      if (moveRec) {
        const float4* rec = reinterpret_cast<const float4*>(recp(i));
        r0 = rec[0];
        r1 = rec[1];
        toi = toip()[i];
      }
      __syncthreads();
      if (keep) {
        cwp()[dst] = w;
        if (moveRec) {
          cpairp()[dst] = pr;
          float4* rec = reinterpret_cast<float4*>(recp(dst));
          rec[0] = r0;
          rec[1] = r1;
          toip()[dst] = toi;
        }
      }
      out += total;
      __syncthreads();
    }
    if (compact && tid == 0) hdr(H_NC) = (uint32_t)out;
    __syncthreads();
  }

  // ------------------------------------------------------------------------------ solver (simple constraints)
  // records: velocity phase rec[2e] = (normal.x, normal.y, normalMass, normalImpulse), rec[2e+1] = (rA.x, rA.y, rB.x, rB.y)
  //          position phase rec[2e] = (localNormal, localPoint),                       rec[2e+1] = (radiusA, radiusB, type, -)
  __device__ __forceinline__ void initSimple(int e) const {
    const uint32_t bb = ent0(e);
    const int bA = (int)(bb & 0xFFFFu), bB = (int)(bb >> 16);
    const int ci = (int)entC(e);
    const uint32_t pr = cpairp()[ci];
    const int pa = (int)(pr & 0xFFFFu), pb = (int)(pr >> 16);
    const float4* rec = reinterpret_cast<const float4*>(recp(ci));
    const float4 r0 = rec[0], r1 = rec[1];
    const int type = (int)(f2u(r1.z) & 0xFFu);
    const float radiusA = __ldg(&px[pa].radius), radiusB = __ldg(&px[pb].radius);
    const float4 cA4 = pos4(bA), cB4 = pos4(bB);
    const float2 kA = massOf(bA), kB = massOf(bB);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    const V2 cA = mk(cA4.x, cA4.y), cB = mk(cB4.x, cB4.y);
    Xf xfA, xfB;
    const float2 qa = q2(bA), qb = q2(bB);
    xfA.q.s = qa.x; xfA.q.c = qa.y;
    xfB.q.s = qb.x; xfB.q.c = qb.y;
    xfA.p = cA - rmul(xfA.q, mk(0.0f, 0.0f));
    xfB.p = cB - rmul(xfB.q, mk(0.0f, 0.0f));
    V2 normal, pt;
    const V2 lp = mk(r0.z, r0.w), ln = mk(r0.x, r0.y);
    const V2 mp0 = mk(0.0f, 0.0f);
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
    rec4(3 * e) = make_float4(normal.x, normal.y, nMass, r1.x);
    rec4(3 * e + 1) = make_float4(rA.x, rA.y, rB.x, rB.y);
    rec4(3 * e + 2) = make_float4(mA, iA, mB, iB);
  }
  // The *Core forms take the schedule entry and the records as values: the relay (below) fetches them from L2 ahead of
  // the warp's turn, so that only the shared-memory traffic on the bodies and the arithmetic are on the critical path.
  // (sA / sB: the two bodies' vel4 or pos4 rows; wA / wB: where the results go -- the same rows, or the dummy row when body A
  //  is the table or when the lane only keeps step with its warp)
  __device__ __forceinline__ void warmStartCore(SF4 sA, SF4 sB, SF4 wA, SF4 wB, const float4& r0, const float4& r1, const float4& r2) const {
    const float2 kA = make_float2(r2.x, r2.y), kB = make_float2(r2.z, r2.w);
    float4 vA = sA, vB = sB;
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
    wA = vA;
    wB = vB;
  }
  __device__ __forceinline__ void warmStartSimple(int e) const {
    const uint32_t bb = ent0(e);
    const SF4 sA = vel4((int)(bb & 0xFFFFu)), sB = vel4((int)(bb >> 16));
    warmStartCore(sA, sB, (int)(bb & 0xFFFFu) != S ? sA : dummy4(), sB, rec4(3 * e), rec4(3 * e + 1), rec4(3 * e + 2));
  }
  // returns the accumulated normal impulse (the caller keeps it in rec4(3e).w)
  __device__ __forceinline__ float solveVelocityCore(SF4 sA, SF4 sB, SF4 wA, SF4 wB, const float4& r0, const float4& r1, const float4& r2) const {
    const float2 kA = make_float2(r2.x, r2.y), kB = make_float2(r2.z, r2.w);
    float4 a4 = sA, b4 = sB;
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
    wA = a4;
    wB = b4;
    return newImpulse;
  }
  __device__ __forceinline__ void solveVelocitySimple(int e) const {
    const uint32_t bb = ent0(e);
    const SF4 sA = vel4((int)(bb & 0xFFFFu)), sB = vel4((int)(bb >> 16));
    rec4(3 * e).set(3, solveVelocityCore(sA, sB, (int)(bb & 0xFFFFu) != S ? sA : dummy4(), sB, rec4(3 * e), rec4(3 * e + 1), rec4(3 * e + 2)));
  }
  // b2ContactSolver::StoreImpulses, then the position-phase records
  __device__ __forceinline__ void storeSimple(int e) const {
    const int ci = (int)entC(e);
    float* rec = recp(ci);
    rec[SR_IMP] = rec4(3 * e).get(3);
    const float4 r0 = reinterpret_cast<const float4*>(rec)[0];
    const uint32_t tp = f2u(rec[SR_TYPE]) & 0xFFu;
    const uint32_t pr = cpairp()[ci];
    rec4(3 * e) = r0;
    rec4(3 * e + 1) = make_float4(__ldg(&px[pr & 0xFFFFu].radius), __ldg(&px[pr >> 16].radius), u2f(tp), 0.0f);
    const int bA = (int)(ent0(e) & 0xFFFFu);
    // kilobot against kilobot: circle manifold, local point zero, local centres zero (no rotation matters)
    if (tp == MANIFOLD_CIRCLES && bA != S && r0.z == 0.0f && r0.w == 0.0f) entI(e) = (uint32_t)entI(e) | 0x8000u;
  }
  // one constraint of b2ContactSolver::SolvePositionConstraints (baumgarte / limit are the regular or the TOI ones)
  __device__ __forceinline__ bool solvePositionSimple(int e, bool fast, float baumgarte, float limit, bool skipZero) const {
    float4 r0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (!fast) r0 = rec4(3 * e);
    const uint32_t bb = ent0(e);
    const SF4 sA = pos4((int)(bb & 0xFFFFu)), sB = pos4((int)(bb >> 16));
    return solvePositionCore(sA, sB, (int)(bb & 0xFFFFu) != S ? sA : dummy4(), sB, fast, r0, rec4(3 * e + 1), rec4(3 * e + 2), baumgarte,
                             limit, skipZero);
  }
  // (r0 is only read when !fast)
  __device__ __forceinline__ bool solvePositionCore(SF4 sA, SF4 sB, SF4 wA, SF4 wB, bool fast, const float4& r0, const float4& r1,
                                                    const float4& r2, float baumgarte, float limit, bool skipZero) const {
    const float2 kA = make_float2(r2.x, r2.y), kB = make_float2(r2.z, r2.w);
    const float mA = kA.x, iA = kA.y, mB = kB.x, iB = kB.y;
    float4 pA4 = sA, pB4 = sB;
    if (fast) {
      float4 a1, b1;
      bool moved, bad = false;
      bool okf = kb_position_pair_t<false>(pA4, pB4, r1.x, r1.y, mA, iA, mB, iB, baumgarte, limit, skipZero, a1, b1, moved, bad);
      if (moved) {
        wA = a1;
        wB = b1;
      }
      if (__builtin_expect(bad, 0)) {   // (off the dependent chain: the rows are stored already)
        okf = kb_position_pair_cold(wA.a, wB.a, pA4, pB4, r1.x, r1.y, mA, iA, mB, iB, baumgarte, limit, skipZero);
      }
      return okf;
    }
    V2 cA = mk(pA4.x, pA4.y), cB = mk(pB4.x, pB4.y);
    V2 normal, point;
    float separation;
    {
      const V2 ln = mk(r0.x, r0.y), lp = mk(r0.z, r0.w);
      const int type = (int)f2u(r1.z);
      // no body of this tier has a local centre or a local manifold point on B: rotations multiply exact zeros
      Xf xfA, xfB;
      xfA.q.s = 0.0f; xfA.q.c = 1.0f;
      xfB.q.s = 0.0f; xfB.q.c = 1.0f;
      xfA.p = cA - rmul(xfA.q, mk(0.0f, 0.0f));
      xfB.p = cB - rmul(xfB.q, mk(0.0f, 0.0f));
      const V2 mpj = mk(0.0f, 0.0f);
      if (type == MANIFOLD_CIRCLES) {
        V2 pointA = xmul(xfA, lp);
        V2 pointB = xmul(xfB, mpj);
        normal = pointB - pointA;
        normalize(normal);
        point = 0.5f * (pointA + pointB);
        separation = dot(pointB - pointA, normal) - r1.x - r1.y;
      } else {
        normal = rmul(xfA.q, ln);
        V2 planePoint = xmul(xfA, lp);
        V2 clipPoint = xmul(xfB, mpj);
        separation = dot(clipPoint - planePoint, normal) - r1.x - r1.y;
        point = clipPoint;
      }
    }
    const bool ok = separation >= limit;
    const float C = b2clamp(baumgarte * (separation + KB_LINEAR_SLOP), -KB_MAX_LINEAR_CORRECTION, 0.0f);
    if (skipZero && C == 0.0f) return ok;   // the impulse is -0 / K and moves nothing
    const V2 rA = point - cA;
    const V2 rB = point - cB;
    const float rnA = cross(rA, normal);
    const float rnB = cross(rB, normal);
    const float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
    const float impulse = K > 0.0f ? -C / K : 0.0f;
    const V2 P = impulse * normal;
    cA = cA - mA * P;
    pA4.z -= iA * cross(rA, P);
    cB = cB + mB * P;
    pB4.z += iB * cross(rB, P);
    pA4.x = cA.x; pA4.y = cA.y;
    wA = pA4;
    pB4.x = cB.x; pB4.y = cB.y;
    wB = pB4;
    return ok;
  }

  // ---- relay: the warps of the CTA take the levels of the schedule in turn, RG levels per turn (turn k = rows RG k ..
  // RG k + RG - 1 belongs to warp k mod NR; the rows of a turn sit in lane groups of RL lanes and are solved one after the
  // other).  A warp fetches its turn's schedule entries and records from L2 while the NR - 1 turns before it are being
  // solved, waits for its predecessor on a named barrier (id 1 + warp; 32 arriving + 32 waiting threads), does the
  // shared-memory part and hands over.  An entry is always solved by the same thread, so its accumulated impulse is
  // thread-private.  (A level wider than RL entries is several rows of the schedule.)
  static constexpr int NR = NT / 32 < 8 ? NT / 32 : 8;
  static constexpr int RG = 4, RL = 32 / RG;
  __device__ __forceinline__ void relayWait(int w) const {
    __syncwarp();
    asm volatile("bar.sync %0, 64;" ::"r"(1 + w) : "memory");
  }
  __device__ __forceinline__ void relayPass(int w) const {
    __syncwarp();   // the warp's shared-memory stores are all issued before it arrives
    asm volatile("bar.arrive %0, 64;" ::"r"(1 + w) : "memory");
  }
  // turn order inside one pass over the turns 0..nTurns-1, repeated without a block-wide barrier in between.  The successor
  // is worked out BEFORE the warp's turn (relayNext), so that the hand-over is one instruction after the last row.  A warp
  // that is its own successor (fewer turns than relay warps, or the wrap-around) arrives on its own barrier and finds the
  // 64 threads complete when it waits.
  __device__ __forceinline__ void relayEnter(int wid, bool firstTurn) const {
    if (!firstTurn) relayWait(wid);
  }
  __device__ __forceinline__ int relayNext(int k, int nTurns) const { return (k == nTurns - 1 ? 0 : k + 1) % NR; }
  __device__ __forceinline__ void relayLeave(int next, bool lastTurn) const {
    if (!lastTurn) relayPass(next);
  }

  // b2World::Solve
  __device__ __forceinline__ void solve() {
    const int nC = (int)hdr(H_NC);
    const int B = L.B;
    uint16_t* const tlC = tlCp();
    const uint32_t tlB = scr(W.sTlB), adj = scr(W.sAdj), bstart = scr(W.sBstart), bcur = scr(W.sBcur);
    const uint32_t ordT = scr(W.sOrd), ordL = scr(W.sOlvl), ordI = scr(W.sOisl), stack = scr(W.sStack);
    // per-body word of the island search: last level (16 bits) | DW_INISLAND | DW_POPPED | DW_AWAKE
    const uint32_t bw = scr(W.sBw), lvlCnt = scr(W.sLvlCnt);
    constexpr uint32_t DW_INISLAND = 1u << 16, DW_POPPED = 1u << 17, DW_AWAKE = 1u << 18;
    // ---- touching list in world-list order (descending contact index)
#pragma unroll 1
    for (int b = tid; b <= B + 1; b += NT) {
      sts_u16(bstart + 2u * (uint32_t)b, 0u);
      if (b <= B) isl(b) = SW_NOISLAND;
    }
    __syncthreads();
    int K = 0;
#pragma unroll 1
    for (int base = 0; base < nC; base += NT) {
      const int i = nC - 1 - (base + tid);
      bool t = false;
      uint32_t bodies = 0u;
      if (i >= 0) {
        const uint32_t w = cwp()[i];
        t = (w & (CI_TOUCHING | CI_ENABLED)) == (CI_TOUCHING | CI_ENABLED);
        if (t) {
          const uint32_t pr = cpairp()[i];
          bodies = (uint32_t)pbody((int)(pr & 0xFFFFu)) | ((uint32_t)pbody((int)(pr >> 16)) << 16);
        }
      }
      int total;
      const int dst = K + blockExScan(t ? 1 : 0, &total);
      if (t && dst < L.Kmax) {
        tlC[dst] = (uint16_t)i;
        sts_u32(tlB + 4u * (uint32_t)dst, bodies);
      }
      K += total;
    }
    if (K > L.Kmax) {
      if (tid == 0) hdr(H_STATUS) |= KB_STATUS_SOLVER_OVERFLOW;
      K = L.Kmax;
    }
    __syncthreads();
    SW_T(2);
    // ---- per-body lists over the touching list (CSR), each sorted ascending == Box2D's contact-edge list order
    // degree counts: bstart[b + 1] (u16) by shared-memory atomics on the containing 32-bit word
#pragma unroll 1
    for (int t = tid; t < K; t += NT) {
      const uint32_t bb = lds_u32(tlB + 4u * (uint32_t)t);
      const int bA = (int)(bb & 0xFFFFu), bB = (int)(bb >> 16);
      if (bA != S) atomicAddU16(bstart, bA + 1);
      if (bB != S) atomicAddU16(bstart, bB + 1);
    }
#pragma unroll 1
    for (int l = tid; l <= K + 1; l += NT) sts_u16(lvlCnt + 2u * (uint32_t)l, 0u);
    __syncthreads();
    {
      // exclusive scan of the degrees over the bodies (chunks of the CTA's width)
      int run = 0;
#pragma unroll 1
      for (int base = 0; base <= B; base += NT) {
        const int b = base + tid;
        const int deg = b <= B ? (int)lds_u16(bstart + 2u * (uint32_t)(b + 1)) : 0;
        int total;
        const int off = run + blockExScan(deg, &total);
        __syncthreads();
        if (b <= B) {
          sts_u16(bcur + 2u * (uint32_t)b, (uint32_t)off);          // fill cursor of body b
          sts_u16(bstart + 2u * (uint32_t)(b + 1), (uint32_t)(off + deg));   // end of body b == start of b + 1
        }
        run += total;
      }
      if (tid == 0) sts_u16(bstart, 0u);
      __syncthreads();
    }
#pragma unroll 1
    for (int t = tid; t < K; t += NT) {
      const uint32_t bb = lds_u32(tlB + 4u * (uint32_t)t);
      const int bA = (int)(bb & 0xFFFFu), bB = (int)(bb >> 16);
      // entry = touching-list index | other body << 16
      if (bA != S) sts_u32(adj + 4u * atomicAddU16(bcur, bA), (uint32_t)t | ((uint32_t)bB << 16));
      if (bB != S) sts_u32(adj + 4u * atomicAddU16(bcur, bB), (uint32_t)t | ((uint32_t)bA << 16));
    }
    __syncthreads();
    uint32_t lonelyCount = 0u;
#pragma unroll 1
    for (int b = tid; b < B; b += NT) {
      const int s0 = (int)lds_u16(bstart + 2u * (uint32_t)b), s1 = (int)lds_u16(bstart + 2u * (uint32_t)(b + 1));
      for (int i = s0 + 1; i < s1; ++i) {   // insertion sort by list index (degree <= ~8)
        const uint32_t v = lds_u32(adj + 4u * (uint32_t)i);
        int j = i - 1;
        while (j >= s0 && (lds_u32(adj + 4u * (uint32_t)j) & 0xFFFFu) > (v & 0xFFFFu)) {
          sts_u32(adj + 4u * (uint32_t)(j + 1), lds_u32(adj + 4u * (uint32_t)j));
          --j;
        }
        sts_u32(adj + 4u * (uint32_t)(j + 1), v);
      }
      const bool aw = awake(b);
      const bool lonely = s1 == s0 && aw;
      if (lonely) {   // an island of its own (b2World::Solve seeds it and finds nothing to add)
        isl(b) = SW_LONELY;
        lonelyCount += 1u;
      }
      sts_u32(bw + 4u * (uint32_t)b, (aw ? DW_AWAKE : 0u) | (lonely ? DW_INISLAND : 0u));
    }
    {
      int total;
      blockExScan((int)lonelyCount, &total);
      lonelyCount = (uint32_t)total;
    }
    __syncthreads();
    SW_T(3);
    // ---- warp 0: island DFS (b2World::Solve) in Box2D's order + dependency level of every constraint:
    // level = 1 + max(level of the earlier constraints that share a dynamic body); the static table never links levels.
    // The search keeps ONE word per body (its last level and flags; a contact is new exactly when its partner has not
    // been popped yet, which is what Box2D's per-contact island flag says).  The contact edges of the popped body are
    // taken by the lanes side by side: the partners of one body are distinct bodies, the new edges get consecutive slots
    // of the constraint order by ballot rank, and the chain  l_i = max(l_(i-1), lo_i) + 1  over the new edges
    // (l_(-1) = the body's own last level) is  l_i = i + 1 + max(lb, max_(j<=i)(lo_j - j)):  a prefix maximum over the lanes.
    // Partners not yet in an island are pushed in edge order (ballot rank), so the stack pops them as Box2D does.
    if (tid < 32) {
      const int lane = tid;
      const uint32_t ltMask = (1u << lane) - 1u;
      int nOrd = 0, nIslands = 0, maxL = 0;   // (warp-uniform)
#pragma unroll 1
      for (int base = ((B - 1) & ~31); base >= 0; base -= 32) {   // body list order: newest (highest index) first
        for (;;) {
          const int sb = base + lane;
          const uint32_t ws = sb < B ? lds_u32(bw + 4u * (uint32_t)sb) : DW_INISLAND;
          const uint32_t cand = __ballot_sync(0xFFFFFFFFu, (ws & DW_INISLAND) == 0u && (ws & DW_AWAKE) != 0u);
          if (cand == 0u) break;
          const int seed = base + 31 - __clz((int)cand);
          int sp = 1;
          if (lane == seed - base) {
            sts_u16(stack, (uint32_t)seed);
            isl(seed) = (uint32_t)nIslands;
            sts_u32(bw + 4u * (uint32_t)seed, ws | DW_INISLAND);
          }
          __syncwarp();
          while (sp > 0) {
            --sp;
            const int b = (int)lds_u16(stack + 2u * (uint32_t)sp);
            const int s0 = (int)lds_u16(bstart + 2u * (uint32_t)b), s1 = (int)lds_u16(bstart + 2u * (uint32_t)(b + 1));
            const uint32_t wb = lds_u32(bw + 4u * (uint32_t)b);
            int lb = (int)(wb & 0xFFFFu);
            if ((wb & DW_AWAKE) == 0u && lane == 0) wake(b);
#pragma unroll 1
            for (int k0 = s0; k0 < s1; k0 += 32) {
              const int k = k0 + lane;
              const bool v = k < s1;
              const uint32_t en = v ? lds_u32(adj + 4u * (uint32_t)k) : 0u;
              const uint32_t t = en & 0xFFFFu, o = en >> 16;
              const bool dyn = v && o != (uint32_t)S;
              const uint32_t wo = dyn ? lds_u32(bw + 4u * o) : 0u;
              const bool isNew = v && !(dyn && (wo & DW_POPPED) != 0u);   // else: added when the partner was popped
              const uint32_t newMask = __ballot_sync(0xFFFFFFFFu, isNew);
              const uint32_t pushMask = __ballot_sync(0xFFFFFFFFu, isNew && dyn && (wo & DW_INISLAND) == 0u);
              if (newMask != 0u) {
                const int r = __popc(newMask & ltMask);
                int val = isNew ? (int)(wo & 0xFFFFu) - r : -0x40000000;
                const int width = s1 - k0;
#pragma unroll 1
                for (int d = 1; d < 32 && d < width; d <<= 1) {
                  const int y = __shfl_up_sync(0xFFFFFFFFu, val, d);
                  if (lane >= d) val = max(val, y);
                }
                const int cnt = __popc(newMask);
                const int l = r + 1 + max(lb, val);
                if (isNew) {
                  const uint32_t slot = (uint32_t)(nOrd + r);
                  sts_u16(ordT + 2u * slot, t);
                  sts_u16(ordL + 2u * slot, (uint32_t)l);
                  sts_u16(ordI + 2u * slot, (uint32_t)nIslands);
                  if (dyn) sts_u32(bw + 4u * o, (wo & ~0xFFFFu) | (uint32_t)l | DW_INISLAND);
                  if (((pushMask >> lane) & 1u) != 0u) {
                    isl((int)o) = (uint32_t)nIslands;
                    sts_u16(stack + 2u * (uint32_t)(sp + __popc(pushMask & ltMask)), o);
                  }
                }
                // the last new edge's level: the highest lane of the chunk holds the maximum over all of them
                lb = cnt + max(lb, __shfl_sync(0xFFFFFFFFu, val, min(width, 32) - 1));
                maxL = max(maxL, lb);
                nOrd += cnt;
                sp += __popc(pushMask);
              }
            }
            if (lane == 0) sts_u32(bw + 4u * (uint32_t)b, (uint32_t)lb | DW_INISLAND | DW_POPPED | DW_AWAKE);
            __syncwarp();
          }
          ++nIslands;
        }
      }
      if (lane == 0) {
        misc(0) = (uint32_t)nOrd;
        misc(2) = (uint32_t)nIslands;
        misc(3) = (uint32_t)maxL;
      }
    }
    __syncthreads();
    const int nOrd = (int)misc(0), nIslDfs = (int)misc(2), maxL = (int)misc(3);
    SW_T(4);
    nIsl += (uint32_t)nIslDfs + lonelyCount;
    nLvl += (uint32_t)maxL;
    // ---- rows: the entries of a level, cut into rows of at most RL (the entries of one level touch disjoint dynamic bodies:
    // their order cannot influence any result, so a wide level may be solved as several rows one after the other).
    // rowStart[r] = first schedule entry of row r, rowStart[nRows] = nOrd; the level's first entry is the scatter cursor.
#pragma unroll 1
    for (int p = tid; p < nOrd; p += NT) atomicAddU16(lvlCnt, (int)lds_u16(ordL + 2u * (uint32_t)p));
    __syncthreads();
    int nRows = 0;
    {
      int run = 0;
#pragma unroll 1
      for (int base = 1; base <= maxL + 1; base += NT) {
        const int l = base + tid;
        const int c = l <= maxL ? (int)lds_u16(lvlCnt + 2u * (uint32_t)l) : 0;
        int total, rtotal;
        const int off = run + blockExScan(c, &total);
        const int nr = (c + RL - 1) / RL;
        const int row = nRows + blockExScan(nr, &rtotal);
        __syncthreads();
        if (l <= maxL + 1) sts_u16(lvlCnt + 2u * (uint32_t)l, (uint32_t)off);   // scatter cursor
        for (int j = 0; j < nr; ++j) rowStart(row + j) = (uint32_t)(off + j * RL);
        run += total;
        nRows += rtotal;
      }
      if (tid == 0) rowStart(nRows) = (uint32_t)nOrd;
      __syncthreads();
    }
    // entries of one level touch disjoint dynamic bodies: their order within the level cannot influence any result
#pragma unroll 1
    for (int p = tid; p < nOrd; p += NT) {
      const int t = (int)lds_u16(ordT + 2u * (uint32_t)p);
      const int l = (int)lds_u16(ordL + 2u * (uint32_t)p);
      const uint32_t e = atomicAddU16(lvlCnt, l);
      ent0((int)e) = lds_u32(tlB + 4u * (uint32_t)t);
      entC((int)e) = (uint32_t)tlC[t];
      entI((int)e) = lds_u16(ordI + 2u * (uint32_t)p);
    }
#pragma unroll 1
    for (int i = tid; i < nIslDfs; i += NT) sts_u8(islStateAddr(i), 1u);   // bit 0: unsolved
    __syncthreads();
    // ---- b2Island::Solve: integrate velocities (damping), remember the sweep start
    const float h = L.dt;
#pragma unroll 1
    for (int b = tid; b < B; b += NT) {
      if ((uint32_t)isl(b) == SW_NOISLAND) continue;
      const float4 p = pos4(b);
      sweepp()[b] = make_float4(p.x, p.y, p.z, 0.0f);
      float4 v = vel4(b);
      const float ld = __ldg(&bc[b].linearDamping), ad = __ldg(&bc[b].angularDamping);
      const float dl = L.dampingMode == 0 ? 1.0f / (1.0f + h * ld) : b2clamp(1.0f - h * ld, 0.0f, 1.0f);
      const float da = L.dampingMode == 0 ? 1.0f / (1.0f + h * ad) : b2clamp(1.0f - h * ad, 0.0f, 1.0f);
      v.x *= dl;
      v.y *= dl;
      v.z *= da;
      vel4(b) = v;
    }
    __syncthreads();   // the schedule is complete: the scratch lists are dead, the record region is free
#pragma unroll 1
    for (int e = tid; e < nOrd; e += NT) initSimple(e);
    nPts += (uint32_t)nOrd;
    __syncthreads();
    SW_T(5);
    // ---- warm start (pass 0) + velocity iterations: the relay over the levels
    const int nTurns = (nRows + RG - 1) / RG;
    {
      const int lane = tid & 31, wid = tid >> 5;
      const int g = lane / RL, li = lane % RL;
      const int passes = 1 + L.velIters;
      if (wid < NR) {
        for (int pass = 0; pass < passes; ++pass) {
#pragma unroll 1
          for (int k = wid; k < nTurns; k += NR) {
            const int row = RG * k + g;
            int s0 = 0, s1 = 0;
            if (row < nRows) {
              s0 = (int)rowStart(row);
              s1 = (int)rowStart(row + 1);
            }
            const int e = s0 + li;
            const bool mine = e < s1;
            const float4 z4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            float4 r0 = z4, r1 = z4, r2 = z4;
            const SF4 dm = dummy4();
            SF4 sA = dm, sB = dm, wA = dm;
            if (mine) {
              const uint32_t bb = ent0(e);
              r0 = rec4(3 * e);
              r1 = rec4(3 * e + 1);
              r2 = rec4(3 * e + 2);
              sA = vel4((int)(bb & 0xFFFFu));
              sB = vel4((int)(bb >> 16));
              if ((int)(bb & 0xFFFFu) != S) wA = sA;
            }
            // the rows every step loads from and stores to (the lane's own in its group's step, the dummy row otherwise):
            // selected here, off the dependent chain
            uint32_t aS[RG], bS[RG], cS[RG];
#pragma unroll
            for (int gg = 0; gg < RG; ++gg) {
              const bool act = g == gg;
              aS[gg] = act ? sA.a : dm.a;
              bS[gg] = act ? sB.a : dm.a;
              cS[gg] = act ? wA.a : dm.a;
            }
            const int nextW = relayNext(k, nTurns);
            relayEnter(wid, pass == 0 && k == 0);
            // the levels of the turn, one after the other: every lane runs every step (no branches on the way), the lanes
            // outside the step's group on the dummy row
            float imp = 0.0f;
            if (pass == 0) {   // (one uniform branch per turn, not per step)
#pragma unroll
              for (int gg = 0; gg < RG; ++gg) {
                warmStartCore(SF4{aS[gg]}, SF4{bS[gg]}, SF4{cS[gg]}, SF4{bS[gg]}, r0, r1, r2);
                __syncwarp();
              }
            } else {
#pragma unroll
              for (int gg = 0; gg < RG; ++gg) {
                const float ni = solveVelocityCore(SF4{aS[gg]}, SF4{bS[gg]}, SF4{cS[gg]}, SF4{bS[gg]}, r0, r1, r2);
                imp = g == gg ? ni : imp;
                __syncwarp();
              }
            }
            relayLeave(nextW, pass == passes - 1 && k == nTurns - 1);
            if (mine && pass != 0) rec4(3 * e).set(3, imp);
          }
        }
      }
    }
    __syncthreads();
    SW_T(6);
#pragma unroll 1
    for (int e = tid; e < nOrd; e += NT) storeSimple(e);
    // ---- integrate positions
#pragma unroll 1
    for (int b = tid; b < B; b += NT) {
      if ((uint32_t)isl(b) == SW_NOISLAND) continue;
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
    __syncthreads();
    SW_T(7);
    // ---- position iterations with per-island early exit (islState bit 0: still iterating, bit 1: a separation
    //      below -3 linearSlop seen in this sweep)
    nPit += (uint32_t)nIslDfs + lonelyCount;   // first iteration of every island (a lonely island is solved by it)
    for (int it = 0; it < L.posIters; ++it) {
      {
        const int lane = tid & 31, wid = tid >> 5;
        const int g = lane / RL, li = lane % RL;
        if (wid < NR) {
#pragma unroll 1
          for (int k = wid; k < nTurns; k += NR) {
            const int row = RG * k + g;
            int s0 = 0, s1 = 0;
            if (row < nRows) {
              s0 = (int)rowStart(row);
              s1 = (int)rowStart(row + 1);
            }
            const int e = s0 + li;
            uint32_t ei = 0x8000u;
            const float4 z4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            float4 r0 = z4, r1 = z4, r2 = z4;
            const SF4 dm = dummy4();
            SF4 sA = dm, sB = dm, wA = dm;
            bool mine = e < s1;
            if (mine) {
              ei = entI(e);
              // (bit 0 of the island's state does not change during a sweep)
              mine = (lds_u8(islStateAddr((int)(ei & 0x7FFFu))) & 1u) != 0u;
            }
            if (mine) {
              const uint32_t bb = ent0(e);
              if ((ei & 0x8000u) == 0u) r0 = rec4(3 * e);
              r1 = rec4(3 * e + 1);
              r2 = rec4(3 * e + 2);
              sA = pos4((int)(bb & 0xFFFFu));
              sB = pos4((int)(bb >> 16));
              if ((int)(bb & 0xFFFFu) != S) wA = sA;
            }
            // (everything a row-step needs besides the two body rows is in registers before the warp's turn: also the
            //  address of the island's state byte and the constant stored there)
            const uint32_t islA = islStateAddr((int)(ei & 0x7FFFu)), three = 3u;
            const bool fastE = (ei & 0x8000u) != 0u;
            const int nextW = relayNext(k, nTurns);
            relayEnter(wid, k == 0);
#ifdef KB_PROFILE
            const long long tr1 = clock64();
#endif
#pragma unroll
            for (int gg = 0; gg < RG; ++gg) {
              // (one guard is cheaper here than running the idle lanes on dummy rows: measured 33.2 vs 35.5 ms with the
              //  straight-line arithmetic, 45.1 vs 51.3 ms when the sqrt / division paths of the idle lanes still diverged)
              if (g == gg && mine) {
                const bool ok = solvePositionCore(sA, sB, wA, sB, fastE, r0, r1, r2, KB_BAUMGARTE, -3.0f * KB_LINEAR_SLOP, true);
                if (!ok) sts_u8(islA, three);
              }
              __syncwarp();
            }
#ifdef KB_PROFILE
            const long long tr2 = clock64();
#endif
            relayLeave(nextW, k == nTurns - 1);
#ifdef KB_PROFILE
            (void)tr1;
            (void)tr2;
#endif
          }
        }
      }
      __syncthreads();
      uint32_t still = 0u;
#pragma unroll 1
      for (int i = tid; i < nIslDfs; i += NT) {
        const uint32_t st = lds_u8(islStateAddr(i));
        const uint32_t ns = (st & 2u) != 0u ? 1u : 0u;   // unsolved &= bad
        sts_u8(islStateAddr(i), ns);
        still += ns;
      }
      int total;
      blockExScan((int)still, &total);
      __syncthreads();
      if (total == 0) break;
      if (it + 1 < L.posIters) nPit += (uint32_t)total;
    }
    // islState now: bit 0 set = position NOT solved.  Re-purpose: bit 1 = some body of the island is not ready to sleep
    __syncthreads();
    SW_T(8);
    // ---- copy back: SynchronizeTransform; sleep bookkeeping
#pragma unroll 1
    for (int b = tid; b < B; b += NT) {
      const uint32_t island = isl(b);
      if (island == SW_NOISLAND) continue;
      const float4 p = pos4(b);
      const Rot q = rot_set(p.z);
      q2(b) = make_float2(q.s, q.c);
      if (L.enableSleep) {
        const float4 v = vel4(b);
        const float linTolSqr = KB_LIN_SLEEP_TOL * KB_LIN_SLEEP_TOL;
        const float angTolSqr = KB_ANG_SLEEP_TOL * KB_ANG_SLEEP_TOL;
        float st;
        if (v.z * v.z > angTolSqr || dot(mk(v.x, v.y), mk(v.x, v.y)) > linTolSqr) st = 0.0f;
        else st = p.w + h;
        pos4(b).set(3, st);
        if (!(st >= KB_TIME_TO_SLEEP)) {
          if (island == SW_LONELY) isl(b) = SW_LONELY - 1u;   // lonely and not ready: marked "stay awake" (0xFFFD)
          else atomicOrU8(islStateAddr((int)island), 2u);
        }
      }
    }
    __syncthreads();
    if (L.enableSleep) {
#pragma unroll 1
      for (int b = tid; b < B; b += NT) {
        const uint32_t island = isl(b);
        if (island == SW_NOISLAND) continue;
        bool sleepNow;
        if (island == SW_LONELY) sleepNow = true;            // positionSolved (no constraints) and minSleepTime reached
        else if (island == SW_LONELY - 1u) sleepNow = false;
        else sleepNow = lds_u8(islStateAddr((int)island)) == 0u;
        if (sleepNow) {
          vel4(b) = make_float4(0.0f, 0.0f, 0.0f, u2f(f2u(vel4(b).get(3)) & ~BF_AWAKE));
          pos4(b).set(3, 0.0f);
        }
      }
    }
    __syncthreads();
    SW_T(9);
    synchronizeFixtures(-1);
    SW_T(10);
    findNewContacts();
    SW_T(11);
  }

  // shared-memory u16 / u8 atomics on the containing 32-bit word
  __device__ __forceinline__ uint32_t atomicAddU16(uint32_t base, int idx) const {
    const uint32_t a = base + 2u * (uint32_t)idx;
    const uint32_t sh = (a & 2u) * 8u;
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a & ~3u), "r"(1u << sh) : "memory");
    return (old >> sh) & 0xFFFFu;
  }
  __device__ __forceinline__ void atomicOrU8(uint32_t a, uint32_t v) const {
    const uint32_t sh = (a & 3u) * 8u;
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a & ~3u), "r"(v << sh) : "memory");
  }

  // b2Body::SynchronizeFixtures + b2BroadPhase::MoveProxy for every body that was in an island (only == -1), or for
  // the one body `only` (TOI mini-island; the sweep start was set to the corrected pose by the caller).
  // A kilobot's proxy is a circle at the body origin with zero local centre: aabb(xf) = xf.p -+ r, xf1.p = c0.
  __device__ __forceinline__ void synchronizeFixtures(int only) {
#pragma unroll 1
    for (int b = tid; b < L.B; b += NT) {
      if (only >= 0 ? b != only : (uint32_t)isl(b) == SW_NOISLAND) continue;
      const int p = nWall + b;
      const float4 sw = sweepp()[b];
      const float4 pc = pos4(b);
      const float r = __ldg(&px[p].radius);
      const V2 p1 = mk(sw.x, sw.y) - rmul(Rot{0.0f, 1.0f}, mk(0.0f, 0.0f));
      const V2 p2 = mk(pc.x, pc.y);
      const V2 c1 = p1 + rmul(Rot{0.0f, 1.0f}, mk(0.0f, 0.0f)), c2 = p2 + rmul(Rot{0.0f, 1.0f}, mk(0.0f, 0.0f));
      const V2 lo = mk(b2min(c1.x - r, c2.x - r), b2min(c1.y - r, c2.y - r));
      const V2 hi = mk(b2max(c1.x + r, c2.x + r), b2max(c1.y + r, c2.y + r));
      const V2 displacement = p2 - p1;
      const float4 fat = fatp()[p];
      const bool contains = fat.x <= lo.x && fat.y <= lo.y && hi.x <= fat.z && hi.y <= fat.w;
      if (!contains) {
        float4 nb = make_float4(lo.x - KB_AABB_EXTENSION, lo.y - KB_AABB_EXTENSION, hi.x + KB_AABB_EXTENSION,
                                hi.y + KB_AABB_EXTENSION);
        const V2 d = KB_AABB_MULTIPLIER * displacement;
        if (d.x < 0.0f) nb.x += d.x; else nb.z += d.x;
        if (d.y < 0.0f) nb.y += d.y; else nb.w += d.y;
        fatp()[p] = nb;
        moved(p >> 5).atomOr(1u << (p & 31));
      }
    }
    __syncthreads();
  }

  // ------------------------------------------------------------------------------ broadphase (uniform grid)
  __device__ __forceinline__ bool isMoved(int p) const { return ((uint32_t)moved(p >> 5) >> (p & 31)) & 1u; }
  __device__ __forceinline__ int cellOf(float c, float origin, int n) const {
    const int k = (int)floorf((c - origin) * W.invCell);
    return k < 0 ? 0 : (k >= n ? n - 1 : k);
  }
  __device__ __forceinline__ bool hashHas(const uint32_t* table, uint32_t key) const {
    uint32_t h = (key * 2654435761u) >> W.hashShift;
    for (;;) {
      const uint32_t k = __ldcg(table + h);   // filled by atomics at L2: read there
      if (k == key) return true;
      if (k == 0u) return false;
      h = (h + 1u) & (uint32_t)(W.hashSize - 1);
    }
  }
  // candidate test for the ordered pair (i < j), both dynamic proxies; fi = fat AABB of i
  __device__ __forceinline__ bool newPair(const uint32_t* table, int i, int j, const float4& fi, bool movedI) const {
    if (!movedI && !isMoved(j)) return false;
    const float4 fj = lds_f4(scr(W.gFat) + 16u * (uint32_t)j);   // (staged by findNewContacts)
    const bool overlap = !(fj.x - fi.z > 0.0f || fj.y - fi.w > 0.0f || fi.x - fj.z > 0.0f || fi.y - fj.w > 0.0f);
    if (!overlap) return false;
    return !hashHas(table, (((uint32_t)i << 16) | (uint32_t)j) + 1u);
  }

  // b2BroadPhase::UpdatePairs + b2ContactManager::AddPair.  New pairs are appended in (min proxy, max proxy) order.
  __device__ __forceinline__ void findNewContacts() {
    const int P = nP;   // (the inert slots of a smaller scene are never binned: their centre lands in a real cell)
    bool any = false;
    for (int w = tid; w < W.movedWords; w += NT) any |= (uint32_t)moved(w) != 0u;
    if (__syncthreads_or(any) == 0) return;
    int nC = (int)hdr(H_NC);
    uint32_t* const table = hashp();
    const uint32_t cellStart = scr(W.gCellStart), cellCur = scr(W.gCellCur), sorted = scr(W.gSorted);
    const uint32_t pcnt = scr(W.gPcnt);
    const int ncell = W.gx * W.gy;
    // ---- hash of the existing pairs; cell counts
    for (int i = tid; i < W.hashSize; i += NT) table[i] = 0u;
    for (int c = tid; c <= ncell; c += NT) sts_u32(cellStart + 4u * (uint32_t)c, 0u);
    __syncthreads();
#pragma unroll 1
    for (int i = tid; i < nC; i += NT) {
      const uint32_t pr = cpairp()[i];
      const uint32_t pa = pr & 0xFFFFu, pb = pr >> 16;
      const uint32_t key = ((pa < pb ? pa : pb) << 16 | (pa < pb ? pb : pa)) + 1u;
      uint32_t h = (key * 2654435761u) >> W.hashShift;
      for (;;) {
        const uint32_t old = atomicCAS(table + h, 0u, key);
        if (old == 0u || old == key) break;
        h = (h + 1u) & (uint32_t)(W.hashSize - 1);
      }
    }
    // dynamic proxies into cells by the centre of their fat AABB; the widest one sets the search radius.
    // Warp-aggregated counting: lanes that hit the same cell are grouped by __match_any_sync, the group's leader
    // adds the group size with one shared-memory atomic, every lane's slot is base + its rank in the group mask.
    float wmax = 0.0f;
#pragma unroll 1
    for (int base = nWall; base < P; base += NT) {
      const int p = base + tid;
      const bool valid = p < P;
      int cell = -1;
      if (valid) {
        const float4 f = fatp()[p];
        wmax = b2max(wmax, b2max(f.z - f.x, f.w - f.y));
        cell = cellOf(0.5f * (f.x + f.z), W.gx0, W.gx) + W.gx * cellOf(0.5f * (f.y + f.w), W.gy0, W.gy);
      }
      const uint32_t act = __ballot_sync(0xFFFFFFFFu, valid);
      if (valid) {
        const uint32_t grp = __match_any_sync(act, cell);
        const int leader = __ffs(grp) - 1, rank = __popc(grp & ((1u << (tid & 31)) - 1u));
        uint32_t slot = 0u;
        if ((tid & 31) == leader)
          asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(slot) : "r"(cellStart + 4u * (uint32_t)(cell + 1)), "r"((uint32_t)__popc(grp)) : "memory");
        slot = __shfl_sync(grp, slot, leader) + (uint32_t)rank;
        sts_u32(pcnt + 4u * (uint32_t)p, ((uint32_t)cell << 12) | slot);   // cell | slot within the cell
      }
    }
    {
      // search radius in cells: two AABBs overlap only if their centres are within (w_i + w_j) / 2 <= wmax per axis
      const float wm = blockMaxF(wmax);
      const int rad = max(1, (int)ceilf(wm * W.invCell));
      if (tid == 0) misc(4) = (uint32_t)rad;
    }
    // exclusive scan of the cell counts (cellStart[c + 1] holds count of cell c)
    {
      int run = 0;
#pragma unroll 1
      for (int base = 0; base < ncell; base += NT) {
        const int c = base + tid;
        const int n = c < ncell ? (int)lds_u32(cellStart + 4u * (uint32_t)(c + 1)) : 0;
        int total;
        const int off = run + blockExScan(n, &total);
        __syncthreads();
        if (c < ncell) sts_u32(cellStart + 4u * (uint32_t)(c + 1), (uint32_t)(off + n));
        run += total;
      }
      __syncthreads();
    }
    for (int p = nWall + tid; p < P; p += NT) {
      const uint32_t cs = lds_u32(pcnt + 4u * (uint32_t)p);
      sts_u16(sorted + 2u * (lds_u32(cellStart + 4u * (cs >> 12)) + (cs & 0xFFFu)), (uint32_t)p);
    }
    // every proxy's fat AABB into shared memory: each is read by ~27 candidate tests (two passes), from L2 otherwise
    for (int p = tid; p < P; p += NT) sts_f4(scr(W.gFat) + 16u * (uint32_t)p, fatp()[p]);
    __syncthreads();
    const int rad = (int)misc(4);
    uint32_t tests = 0u;
    bool overflow = false;
#ifdef KB_PROFILE
    __syncthreads();
    const long long tf0 = clock64();
    tp[14] += tf0 - tlast;   // (find new contacts: pair hash + grid build)
#endif
    // ---- table edges first (lowest proxy ids): every dynamic proxy j against edge i, block-wide
    for (int i = 0; i < nWall; ++i) {
      const float4 fi = fatp()[i];
      const bool movedI = isMoved(i);
#pragma unroll 1
      for (int base = nWall; base < P; base += NT) {
        const int j = base + tid;
        bool c = false;
        if (j < P && (movedI || isMoved(j))) {
          tests += 1u;
          c = newPair(table, i, j, fi, true);
        }
        int total;
        const int dst = nC + blockExScan(c ? 1 : 0, &total);
        if (c) {
          if (dst < L.Cmax) {
            cwp()[dst] = CI_ENABLED;
            cpairp()[dst] = (uint32_t)i | ((uint32_t)j << 16);   // chain edge takes the A slot (b2Contact::Create)
            toip()[dst] = 1.0f;
            wake(pbody(j));
          } else {
            overflow = true;
          }
        }
        nC = min(nC + total, L.Cmax);
      }
    }
#ifdef KB_PROFILE
    __syncthreads();
    (void)tf0;
#endif
    // ---- dynamic against dynamic through the grid: proxy i owns its pairs (i, j > i).
    // The walk over the (2 rad + 1)^2 cells is WARP-COHERENT: every lane takes the same number of cells (clipped ones are
    // empty ranges) and the warp's widest cell sets the inner trip count, so the lanes stay on one path through the loads
    // and comparisons and only the hash look-up of an overlapping pair diverges (with each lane walking its own ragged
    // ranges the warp serialised up to 32 different paths: 0.45 of 0.5 Mcycles per sub-step at 1024 kilobots).
    // The walk only COLLECTS the partners whose fat AABBs overlap (at most KB_SW_CAND per proxy in a per-thread row of
    // shared memory); whether such a pair already has a contact is then asked of the L2-resident hash for all of them at
    // once (independent loads in flight together: one L2 round trip per proxy instead of one per candidate, on a path the
    // whole warp waits on), and the new ones are emitted in ascending order from the same row -- no second walk.
    constexpr int KB_SW_CAND = 12;
    const uint32_t candRow = scr(W.gCand) + 2u * (uint32_t)(KB_SW_CAND * tid);
    const int side = 2 * rad + 1;
#pragma unroll 1
    for (int base = nWall; base < P; base += NT) {
      const int i = base + tid;
      const bool live = i < P;
      float4 fi = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      int cx = 0, cy = 0;
      bool movedI = false;
      if (live) {
        fi = lds_f4(scr(W.gFat) + 16u * (uint32_t)i);
        movedI = isMoved(i);
        cx = cellOf(0.5f * (fi.x + fi.z), W.gx0, W.gx);
        cy = cellOf(0.5f * (fi.y + fi.w), W.gy0, W.gy);
      }
      int nCand = 0, cnt = 0;
#pragma unroll 1
      for (int ci = 0; ci < side * side; ++ci) {
        const int xx = cx - rad + ci % side, yy = cy - rad + ci / side;
        int s0 = 0, s1 = 0;
        if (live && xx >= 0 && xx < W.gx && yy >= 0 && yy < W.gy) {
          const int c = xx + W.gx * yy;
          s0 = (int)lds_u32(cellStart + 4u * (uint32_t)c);
          s1 = (int)lds_u32(cellStart + 4u * (uint32_t)(c + 1));
        }
        const int nmax = (int)__reduce_max_sync(0xFFFFFFFFu, (uint32_t)(s1 - s0));
#pragma unroll 1
        for (int t = 0; t < nmax; ++t) {
          const bool v = s0 + t < s1;
          const int j = v ? (int)lds_u16(sorted + 2u * (uint32_t)(s0 + t)) : 0;
          bool cand = v && j > i && (movedI || isMoved(j));
          if (cand) {
            tests += 1u;
            const float4 fj = lds_f4(scr(W.gFat) + 16u * (uint32_t)j);
            cand = !(fj.x - fi.z > 0.0f || fj.y - fi.w > 0.0f || fi.x - fj.z > 0.0f || fi.y - fj.w > 0.0f);
          }
          if (cand) {
            if (nCand < KB_SW_CAND) sts_u16(candRow + 2u * (uint32_t)nCand, (uint32_t)j);
            ++nCand;   // (more than the row holds: the plain walk below)
          }
        }
      }
      // first probe of every collected pair, all in flight together; a collision continues the probe sequence
      uint32_t isNew = 0u;
      {
        uint32_t probe[KB_SW_CAND], slot[KB_SW_CAND], key[KB_SW_CAND];
#pragma unroll
        for (int q = 0; q < KB_SW_CAND; ++q) {
          const uint32_t j = q < nCand ? lds_u16(candRow + 2u * (uint32_t)q) : 0u;
          key[q] = (((uint32_t)i << 16) | j) + 1u;
          slot[q] = (key[q] * 2654435761u) >> W.hashShift;
          probe[q] = q < nCand ? __ldcg(table + slot[q]) : key[q];
        }
#pragma unroll
        for (int q = 0; q < KB_SW_CAND; ++q) {
          if (q < nCand && probe[q] != key[q]) {
            bool found = false;
            uint32_t k = probe[q], h = slot[q];
            while (k != 0u) {
              h = (h + 1u) & (uint32_t)(W.hashSize - 1);
              k = __ldcg(table + h);
              if (k == key[q]) {
                found = true;
                break;
              }
            }
            if (!found) isNew |= 1u << q;
          }
        }
      }
      const bool rowFull = nCand > KB_SW_CAND;   // more overlapping partners than the row holds
      nCand = min(nCand, KB_SW_CAND);
      cnt = __popc(isNew);
#ifdef KB_PROFILE
      const long long tg0 = clock64();
#endif
      if (rowFull) {
        // (never at the densities a table holds: a fat AABB overlaps a dozen others only in a heap of stacked spawns)
        // count and emit by the plain walk: repeated selection of the smallest new partner above the last one
        cnt = 0;
        for (int yy = max(cy - rad, 0); yy <= min(cy + rad, W.gy - 1); ++yy)
          for (int xx = max(cx - rad, 0); xx <= min(cx + rad, W.gx - 1); ++xx) {
            const int c = xx + W.gx * yy;
            const int s0 = (int)lds_u32(cellStart + 4u * (uint32_t)c), s1 = (int)lds_u32(cellStart + 4u * (uint32_t)(c + 1));
            for (int k = s0; k < s1; ++k) {
              const int j = (int)lds_u16(sorted + 2u * (uint32_t)k);
              if (j > i && newPair(table, i, j, fi, movedI)) ++cnt;
            }
          }
      }
      int total;
      int dst = nC + blockExScan(cnt, &total);
#ifdef KB_PROFILE
      tp[15] += clock64() - tg0;   // (find new contacts: thread 0 waiting for the slowest thread's candidate tests)
#endif
      if (cnt > 0) {
        wake(pbody(i));
        // emit the partners in ascending order: repeated selection of the smallest new j above the last one
        int last = i;
        for (int n = 0; n < cnt; ++n) {
          int best = 0x7FFFFFFF;
          if (!rowFull) {
            for (int q = 0; q < nCand; ++q) {
              const int j = (int)lds_u16(candRow + 2u * (uint32_t)q);
              if (((isNew >> q) & 1u) != 0u && j > last && j < best) best = j;
            }
          } else {
            for (int yy = max(cy - rad, 0); yy <= min(cy + rad, W.gy - 1); ++yy)
              for (int xx = max(cx - rad, 0); xx <= min(cx + rad, W.gx - 1); ++xx) {
                const int c = xx + W.gx * yy;
                const int s0 = (int)lds_u32(cellStart + 4u * (uint32_t)c), s1 = (int)lds_u32(cellStart + 4u * (uint32_t)(c + 1));
                for (int k = s0; k < s1; ++k) {
                  const int j = (int)lds_u16(sorted + 2u * (uint32_t)k);
                  if (j > last && j < best && newPair(table, i, j, fi, movedI)) best = j;
                }
              }
          }
          if (dst < L.Cmax) {
            cwp()[dst] = CI_ENABLED;
            cpairp()[dst] = (uint32_t)i | ((uint32_t)best << 16);
            toip()[dst] = 1.0f;
            wake(pbody(best));
          } else {
            overflow = true;
          }
          last = best;
          ++dst;
        }
      }
      nC = min(nC + total, L.Cmax);
    }
    {
      int total;
      blockExScan((int)tests, &total);
      nTests += (uint32_t)total;
    }
    const bool ov = __syncthreads_or(overflow) != 0;
    if (tid == 0) {
      hdr(H_NC) = (uint32_t)nC;
      if (ov) hdr(H_STATUS) |= KB_STATUS_CONTACT_OVERFLOW;
    }
    for (int w = tid; w < W.movedWords; w += NT) moved(w) = 0u;
    __syncthreads();
  }
  __device__ __forceinline__ float blockMaxF(float v) const {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = b2max(v, __shfl_xor_sync(0xFFFFFFFFu, v, d));
    __syncthreads();
    if ((tid & 31) == 0) misc(16 + (tid >> 5)) = f2u(v);
    __syncthreads();
    float r = 0.0f;
    for (int w = 0; w < NT / 32; ++w) r = b2max(r, u2f(misc(16 + w)));
    return r;
  }

  // ------------------------------------------------------------------------------ b2World::SolveTOI
  // Only table-edge-against-kilobot contacts are candidates (no bullets).  Candidate TOIs are computed by one thread
  // each; the event -- a mini island of the one kilobot and its touching wall contacts -- is solved by thread 0.
  __device__ __forceinline__ void solveTOI() {
    const int B = L.B;
    int nC = (int)hdr(H_NC);
    bool wall = false;
#pragma unroll 1
    for (int i = tid; i < nC; i += NT) wall |= (int)(cpairp()[i] & 0xFFFFu) < nWall;
    if (__syncthreads_or(wall) == 0) return;
#pragma unroll 1
    for (int b = tid; b < B; b += NT) reinterpret_cast<float*>(sweepp() + b)[3] = 0.0f;   // alpha0 = 0
#pragma unroll 1
    for (int i = tid; i < nC; i += NT) {
      cwp()[i] &= ~(CI_TOI | CI_TOICOUNT_MASK);
      toip()[i] = 1.0f;
    }
    if (tid == 0) misc(8) = f2u(0.0f);   // the table's alpha0
    __syncthreads();
    for (int guard = 0; guard < 64 * KB_MAX_SUB_STEPS; ++guard) {
      nC = (int)hdr(H_NC);
      const float tableAlpha0 = u2f(misc(8));
      // ---- per-contact TOI; a body lagging behind the table's alpha0 is advanced first (idempotent per body: all of
      //      its wall contacts advance it to the same target, so the first pass advances, the second computes)
#pragma unroll 1
      for (int i = tid; i < nC; i += NT) {
        const uint32_t w = cwp()[i];
        const uint32_t pr = cpairp()[i];
        const int pa = (int)(pr & 0xFFFFu);
        if (pa >= nWall) continue;
        const int toiCount = (w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT;
        if ((w & CI_ENABLED) == 0u || toiCount > KB_MAX_SUB_STEPS || (w & CI_TOI) != 0u) continue;
        const int bd = pbody((int)(pr >> 16));
        if (!awake(bd)) continue;
        float4 sw = sweepp()[bd];
        if (sw.w < tableAlpha0) {
          const float4 p = pos4(bd);
          const float beta = (tableAlpha0 - sw.w) / (1.0f - sw.w);
          sw.x += beta * (p.x - sw.x);
          sw.y += beta * (p.y - sw.y);
          sw.z += beta * (p.z - sw.z);
          sw.w = tableAlpha0;
          sweepp()[bd] = sw;   // several contacts of one body write identical values
        }
      }
      __syncthreads();
#pragma unroll 1
      for (int i = tid; i < nC; i += NT) {
        const uint32_t w = cwp()[i];
        const uint32_t pr = cpairp()[i];
        const int pa = (int)(pr & 0xFFFFu), pb = (int)(pr >> 16);
        if (pa >= nWall) continue;
        const int toiCount = (w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT;
        if ((w & CI_ENABLED) == 0u || toiCount > KB_MAX_SUB_STEPS || (w & CI_TOI) != 0u) continue;
        const int bd = pbody(pb);
        if (!awake(bd)) continue;
        const float4 sw = sweepp()[bd];
        const float4 p = pos4(bd);
        SweepD sA, sB;
        sA.lc = mk(0.0f, 0.0f); sA.c0 = mk(0.0f, 0.0f); sA.c = mk(0.0f, 0.0f);
        sA.a0 = 0.0f; sA.a = 0.0f; sA.alpha0 = tableAlpha0;
        sA.fixedRot = 1;
        sB.lc = mk(0.0f, 0.0f); sB.c0 = mk(sw.x, sw.y); sB.c = mk(p.x, p.y);
        sB.a0 = sw.z; sB.a = p.z; sB.alpha0 = sw.w;
        sB.fixedRot = 1;
        float alpha = 1.0f;
        const float t = time_of_impact_edge_circle(px + pa, sA, px + pb, sB);
        if (t >= 0.0f) alpha = b2min(tableAlpha0 + (1.0f - tableAlpha0) * t, 1.0f);
        toip()[i] = alpha;
        cwp()[i] = w | CI_TOI;
      }
      __syncthreads();
      // ---- minimum alpha, first in world-list order (highest index) on ties: key = alpha bits << 32 | ~index
      unsigned long long best = ~0ull;
#pragma unroll 1
      for (int i = tid; i < nC; i += NT) {
        const uint32_t w = cwp()[i];
        if ((int)(cpairp()[i] & 0xFFFFu) >= nWall) continue;
        const int toiCount = (w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT;
        if ((w & CI_ENABLED) != 0u && toiCount <= KB_MAX_SUB_STEPS && (w & CI_TOI) != 0u) {
          const float alpha = toip()[i];
          if (alpha < 1.0f) {
            const unsigned long long key = ((unsigned long long)f2u(alpha) << 32) | (uint32_t)(0x7FFFFFFF - i);
            best = key < best ? key : best;
          }
        }
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, best, d);
        best = o < best ? o : best;
      }
      __syncthreads();
      if ((tid & 31) == 0) {
        misc(16 + 2 * (tid >> 5)) = (uint32_t)best;
        misc(17 + 2 * (tid >> 5)) = (uint32_t)(best >> 32);
      }
      __syncthreads();
      for (int w = 0; w < NT / 32; ++w) {
        const unsigned long long o = (unsigned long long)(uint32_t)misc(16 + 2 * w) | ((unsigned long long)(uint32_t)misc(17 + 2 * w) << 32);
        best = o < best ? o : best;
      }
      __syncthreads();
      if (best == ~0ull) break;
      const float minAlpha = u2f((uint32_t)(best >> 32));
      const int minContact = 0x7FFFFFFF - (int)(uint32_t)best;
      if (1.0f - 10.0f * KB_EPS < minAlpha) break;
      nToi += 1u;
      const int bd = pbody((int)(cpairp()[minContact] >> 16));
      // ---- the event (thread 0)
      if (tid == 0) {
        const float4 backupSweep = sweepp()[bd], backupPos = pos4(bd);
        const float2 backupQ = q2(bd);
        {
          float4 sw = backupSweep;
          float4 p = backupPos;
          const float beta = (minAlpha - sw.w) / (1.0f - sw.w);
          sw.x += beta * (p.x - sw.x);
          sw.y += beta * (p.y - sw.y);
          sw.z += beta * (p.z - sw.z);
          sw.w = minAlpha;
          p.x = sw.x; p.y = sw.y; p.z = sw.z;
          sweepp()[bd] = sw;
          pos4(bd) = p;
          const Rot q = rot_set(p.z);
          q2(bd) = make_float2(q.s, q.c);
        }
        updateContact(minContact);
        uint32_t w = cwp()[minContact];
        w &= ~CI_TOI;
        const uint32_t tc = ((w & CI_TOICOUNT_MASK) >> CI_TOICOUNT_SHIFT) + 1u;
        w = (w & ~CI_TOICOUNT_MASK) | (tc << CI_TOICOUNT_SHIFT);
        cwp()[minContact] = w;
        if ((w & CI_TOUCHING) == 0u) {
          cwp()[minContact] = w & ~CI_ENABLED;
          sweepp()[bd] = backupSweep;
          pos4(bd) = backupPos;
          q2(bd) = backupQ;
          misc(9) = 0u;   // no event island
        } else {
          misc(8) = f2u(minAlpha);   // the table advanced with the kilobot
          wake(bd);
          // mini island: minContact, then the kilobot's other touching wall contacts in list order (descending
          // index), each re-evaluated at the advanced pose.  Entries 0.. of the schedule arrays are free here.
          const int cap = min(KB_MAX_TOI_CONTACTS, L.Kmax);
          int nIsland = 0;
          ent0(nIsland) = (uint32_t)S | ((uint32_t)bd << 16);
          entC(nIsland) = (uint32_t)minContact;
          ++nIsland;
          for (int i = nC - 1; i >= 0; --i) {
            if (i == minContact) continue;
            const uint32_t pr = cpairp()[i];
            if ((int)(pr & 0xFFFFu) < nWall && pbody((int)(pr >> 16)) == bd) {
              updateContact(i);
              const uint32_t wi = cwp()[i];
              if ((wi & (CI_ENABLED | CI_TOUCHING)) == (CI_ENABLED | CI_TOUCHING) && nIsland < cap) {
                ent0(nIsland) = (uint32_t)S | ((uint32_t)bd << 16);
                entC(nIsland) = (uint32_t)i;
                ++nIsland;
              }
            }
          }
          // b2Island::SolveTOI: position constraints (TOI baumgarte, -1.5 slop), then velocity constraints without
          // warm starting at the corrected pose, then the remainder of the step
          for (int k = 0; k < nIsland; ++k) {
            const int ci = (int)entC(k);
            const float* rec = recp(ci);
            const float4 r0 = reinterpret_cast<const float4*>(rec)[0];
            const uint32_t pr = cpairp()[ci];
            rec4(3 * k) = r0;
            rec4(3 * k + 2) = make_float4(0.0f, 0.0f, massOf(bd).x, massOf(bd).y);   // the table against the kilobot
            rec4(3 * k + 1) = make_float4(__ldg(&px[pr & 0xFFFFu].radius), __ldg(&px[pr >> 16].radius),
                                          u2f(f2u(rec[SR_TYPE]) & 0xFFu), 0.0f);
          }
          for (int it = 0; it < 20; ++it) {
            bool ok = true;
            for (int k = 0; k < nIsland; ++k) ok &= solvePositionSimple(k, false, KB_TOI_BAUMGARTE, -1.5f * KB_LINEAR_SLOP, false);
            if (ok) break;
          }
          {
            const float4 p = pos4(bd);
            float4 sw = sweepp()[bd];
            sw.x = p.x; sw.y = p.y; sw.z = p.z;
            sweepp()[bd] = sw;
            const Rot q = rot_set(p.z);   // b2ContactSolver rebuilds the transforms from the corrected pose
            q2(bd) = make_float2(q.s, q.c);
          }
          for (int k = 0; k < nIsland; ++k) {
            initSimple(k);
            rec4(3 * k).set(3, 0.0f);   // no warm starting
          }
          for (int it = 0; it < L.velIters; ++it)
            for (int k = 0; k < nIsland; ++k) solveVelocitySimple(k);
          {
            const float h = (1.0f - minAlpha) * L.dt;
            float4 p = pos4(bd);
            float4 v = vel4(bd);
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
            const Rot q = rot_set(p.z);
            q2(bd) = make_float2(q.s, q.c);
          }
          misc(9) = 1u;
        }
      }
      __syncthreads();
      if ((uint32_t)misc(9) == 0u) continue;
      synchronizeFixtures(bd);
      // invalidate the cached TOIs of every contact of the displaced body
#pragma unroll 1
      for (int i = tid; i < nC; i += NT) {
        const uint32_t pr = cpairp()[i];
        if (pbody((int)(pr & 0xFFFFu)) == bd || pbody((int)(pr >> 16)) == bd) cwp()[i] &= ~CI_TOI;
      }
      __syncthreads();
      findNewContacts();
    }
    __syncthreads();
  }

  // b2World::Step(dt, velIters, posIters)
  __device__ __forceinline__ void worldStep() {
    nSub += 1u;
    nCon += hdr(H_NC);
    SW_T(0);
    collide();
    SW_T(1);
    solve();
    if (L.enableToi) solveTOI();
    SW_T(12);
  }

  // ----------------------------------------------------------------------------- outputs
  __device__ __forceinline__ void gather(const KernelArgs& a, int env) {
    __syncthreads();
    const int N = L.N;
    bool bad = false;
    float* flat = a.obsFlat ? a.obsFlat + (size_t)env * (2 * N + L.L) : nullptr;
#pragma unroll 1
    for (int b = tid; b < L.B; b += NT) {
      float4 p = pos4(b);
      float ox = (float)((double)p.x / 25.0), oy = (float)((double)p.y / 25.0);
      if (b >= nP - nWall) {   // absent kilobot (kilobots only: body b owns proxy nWall + b): quiet NaN rows
        ox = oy = p.z = __int_as_float(0x7FC00000);
      } else {
        bad |= !(isfinite(p.x) && isfinite(p.y) && isfinite(p.z));
      }
      if (a.obsKilobots) {
        float* o = a.obsKilobots + ((size_t)env * N + b) * 3;
        o[0] = ox;
        o[1] = oy;
        o[2] = p.z;
      }
      if (flat) {
        flat[2 * b] = ox;
        flat[2 * b + 1] = oy;
      }
    }
    const bool anyBad = __syncthreads_or(bad) != 0;
    if (anyBad && tid == 0) hdr(H_STATUS) |= KB_STATUS_NONFINITE;
    observeLights(*this, a, env, flat, tid, NT);
    __syncthreads();
    if (tid == 0) taskEnd(*this, a, env);
  }
};

// ----------------------------------------------------------------------------------- kernels
// the scene an env was last reset with (kb_set_env_scene takes effect at the next reset)
__device__ __forceinline__ int swarmSceneOf(const KernelArgs& a, int env) {
  return a.envScene ? (int)reinterpret_cast<const uint32_t*>(a.blobs + (size_t)env * a.L.blobWords)[a.L.oHdr + H_SCENE] : 0;
}

template <int NT>
__device__ __forceinline__ void swarmBind(Swarm<NT>& s, const KernelArgs& a, int env, int scene) {
  s.blob = a.blobs + (size_t)env * a.L.blobWords;
  s.px = a.proxies + (size_t)scene * a.L.Pp;
  s.bc = a.bodies + (size_t)scene * a.L.Bp;
  s.nWall = __ldg(&a.scenes[scene].wallEdges);
  s.nP = __ldg(&a.scenes[scene].numProxies);
}

template <int NT>
__global__ void __launch_bounds__(NT, NT >= 512 ? 1 : (NT >= 256 ? 2 : 4)) kb_swarm_step_kernel(const __grid_constant__ KernelArgs a) {
  const int env = a.envOffset + blockIdx.x;
  Swarm<NT> s(a.L, a.W);
  const int scene = swarmSceneOf(a, env);
  swarmBind(s, a, env, scene);
  s.loadState();
  s.loadConsts(a.lights + (size_t)scene * (a.L.numLights > 0 ? a.L.numLights : 1));
  const int A = a.actionMode == KB_ACTION_KILOBOTS ? 2 * a.L.N : a.L.A;
  const double* act = a.action ? a.action + (size_t)env * A : nullptr;
  if (a.actionMode == KB_ACTION_KILOBOTS) {
    setKilobotActions(s, act, s.tid, NT);
    __syncthreads();
  }
  if (a.task.mode != KB_TASK_CONST && s.tid == 0) taskBegin(s, a, env);
  for (int step = 0; step < a.L.stepsPerAction; ++step) {
    if (a.actionMode == KB_ACTION_LIGHT && act && a.L.numLights > 0) {
      if (s.tid == 0) lightStep(s, act);
      __syncthreads();
    }
    senseControl(s, s.tid, NT);
    __syncthreads();
    s.worldStep();
  }
  s.gather(a, env);
  s.storeState();
#ifdef KB_PROFILE
  s.tp[13] += clock64() - s.tlast;
  if (a.prof && s.tid == 0)
    for (int i = 0; i < KB_PROF_SLOTS; ++i) a.prof[(size_t)env * KB_PROF_SLOTS + i] = (unsigned long long)s.tp[i];
#endif
}

template <int NT>
__global__ void __launch_bounds__(NT, NT >= 512 ? 1 : (NT >= 256 ? 2 : 4)) kb_swarm_reset_kernel(const __grid_constant__ KernelArgs a) {
  const int env = blockIdx.x;
  if (a.mask && !a.mask[env]) return;
  const Layout& L = a.L;
  Swarm<NT> s(a.L, a.W);
  int scene = a.envScene ? a.envScene[env] : 0;
  if (a.sampler) {   // a fresh scene drawn on the device (kb_sample.cuh)
    const uint32_t ep = a.episode[env];
    scene = sampleScene(a, env, scene, ep, s.tid, NT, []() { __syncthreads(); });
    if (s.tid == 0) {
      a.episode[env] = ep + 1u;
      if (a.envSceneW) a.envSceneW[env] = scene;
    }
    __syncthreads();
  }
  swarmBind(s, a, env, scene);
  const int tid = s.tid;
  uint32_t* bw = reinterpret_cast<uint32_t*>(s.blob);
  for (int i = tid; i < 2 * KB_NUM_COUNTERS; i += NT) bw[L.oCnt + i] = 0u;
  for (int i = tid; i < H_WORDS; i += NT) s.hdr(i) = 0u;
  __syncthreads();
  if (tid == 0) s.hdr(H_SCENE) = (uint32_t)scene;
  resetEnvLayer(s, a, env, env, tid, NT);
  for (int b = tid; b <= L.B; b += NT) {
    if (b < s.nP - s.nWall) {
      const double* p = a.pose + ((size_t)env * L.B + b) * 3;
      const float x = (float)(25.0 * p[0]);
      const float y = (float)(25.0 * p[1]);
      const float ang = (float)p[2];
      const Rot q = rot_set(ang);
      s.pos4(b) = make_float4(x, y, ang, 0.0f);
      s.vel4(b) = make_float4(0.0f, 0.0f, 0.0f, u2f(BF_AWAKE));
      s.q2(b) = make_float2(q.s, q.c);
      s.sweepp()[b] = make_float4(x, y, ang, 0.0f);
    } else {
      // the static slot B, and any absent body (a padded index the scene does not populate) in the canonical state:
      // zero pose and velocity, asleep, identity transform
      s.pos4(b) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      s.vel4(b) = make_float4(0.0f, 0.0f, 0.0f, b == L.B ? u2f(BF_AWAKE) : 0.0f);
      s.q2(b) = make_float2(0.0f, 1.0f);
      if (b < L.B) s.sweepp()[b] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
  }
  s.loadConsts(a.lights + (size_t)scene * (L.numLights > 0 ? L.numLights : 1));
  // proxies: b2Fixture::CreateProxies -> fat AABB = aabb -+ aabbExtension, every proxy buffered as moved
  for (int w = tid; w < a.W.movedWords; w += NT) s.moved(w) = 0u;
  __syncthreads();
  for (int p = tid; p < L.P; p += NT) {
    float4 f;
    if (p < s.nWall) {
      const V2 v1 = pvert(s.px + p, 1), v2 = pvert(s.px + p, 2);
      const Xf id = Xf{mk(0.0f, 0.0f), Rot{0.0f, 1.0f}};
      const V2 p1 = xmul(id, v1), p2 = xmul(id, v2);
      f = make_float4(b2min(p1.x, p2.x) - KB_AABB_EXTENSION, b2min(p1.y, p2.y) - KB_AABB_EXTENSION,
                      b2max(p1.x, p2.x) + KB_AABB_EXTENSION, b2max(p1.y, p2.y) + KB_AABB_EXTENSION);
    } else if (p < s.nP) {
      const Xf xf = s.bodyXf(p - s.nWall);
      const float r = __ldg(&s.px[p].radius);
      const V2 cc = xf.p + rmul(xf.q, mk(0.0f, 0.0f));   // b2CircleShape::ComputeAABB
      f = make_float4((cc.x - r) - KB_AABB_EXTENSION, (cc.y - r) - KB_AABB_EXTENSION, (cc.x + r) + KB_AABB_EXTENSION,
                      (cc.y + r) + KB_AABB_EXTENSION);
    } else {
      f = make_float4(3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f);
    }
    s.fatp()[p] = f;
    if (p < s.nP) s.moved(p >> 5).atomOr(1u << (p & 31));
  }
  __syncthreads();
  s.findNewContacts();   // b2World::Step: m_flags & e_newFixture -> FindNewContacts
  s.worldStep();         // kilobots_env.py:157 "step to resolve"
  if (tid == 0 && a.status) a.status[env] = (int32_t)s.hdr(H_STATUS);
  s.storeState();
}

// Body.set_pose (lib/body.py:67-69) -> b2Body::SetTransform on the flagged bodies
template <int NT>
__global__ void __launch_bounds__(NT, NT >= 512 ? 1 : (NT >= 256 ? 2 : 4)) kb_swarm_setpose_kernel(const __grid_constant__ KernelArgs a) {
  const int env = blockIdx.x;
  const Layout& L = a.L;
  Swarm<NT> s(a.L, a.W);
  swarmBind(s, a, env, swarmSceneOf(a, env));
  s.loadState();
  for (int b = s.tid; b < s.nP - s.nWall; b += NT) {   // (absent bodies are left alone)
    if (a.mask && !a.mask[(size_t)env * L.B + b]) continue;
    const double* p = a.pose + ((size_t)env * L.B + b) * 3;
    const float x = (float)(p[0] * 25.0);
    const float y = (float)(p[1] * 25.0);
    const float ang = (float)p[2];
    const Rot q = rot_set(ang);
    float4 pos = s.pos4(b);
    pos.x = x; pos.y = y; pos.z = ang;
    s.pos4(b) = pos;
    s.q2(b) = make_float2(q.s, q.c);
    s.sweepp()[b] = make_float4(x, y, ang, 0.0f);
    // SetTransform: Synchronize(xf, xf), zero displacement
    const int pr = s.nWall + b;
    const float r = __ldg(&s.px[pr].radius);
    const float4 fat = s.fatp()[pr];
    const V2 lo = mk(x - r, y - r), hi = mk(x + r, y + r);
    const bool contains = fat.x <= lo.x && fat.y <= lo.y && hi.x <= fat.z && hi.y <= fat.w;
    if (!contains) {
      s.fatp()[pr] = make_float4(lo.x - KB_AABB_EXTENSION, lo.y - KB_AABB_EXTENSION, hi.x + KB_AABB_EXTENSION,
                                 hi.y + KB_AABB_EXTENSION);
      s.moved(pr >> 5).atomOr(1u << (pr & 31));
    }
  }
  s.storeState();
}

}  // namespace kb
