/*
 * kb_b200.h -- C-ABI of the B200-native batched Kilobots step.
 *
 * Drop-in boundary for the hot path of gregorgebhardt/gym-kilobots: KilobotsEnv.step
 * (reference: gym_kilobots/envs/kilobots_env.py:161-215) and KilobotsEnv.reset (:150-159).
 * The reference has no FFI of its own; its only native boundary is pybox2d's per-object
 * SWIG API (b2World.Step at kilobots_env.py:187/:218, b2Body property get/set at
 * lib/body.py:32-38,63-65, lib/kilobot.py:111-127,201-203,254-258).  This header is the
 * batched replacement for that whole call pattern: one call steps E environments.
 *
 * Conventions
 *   - plain C, no torch types.  Every function returns 0 on success or a negative KbError;
 *     kb_last_error() returns the message of the last failure on the calling thread.
 *   - "b2 units" = metres * 25 (lib/body.py:7).  Geometry in the scene description is in
 *     b2 units, float32, exactly as the reference hands it to Box2D; poses, light state and
 *     actions cross the boundary in SI units (metres, radians), float64, as the reference's
 *     numpy arrays do.
 *   - the same entry points exist with the prefix kbo_ in oracle/libkbo.so (CPU oracle; test
 *     infrastructure only) taking HOST pointers everywhere, so tests drive both identically.
 *   - kb_* functions taking "device pointer" arguments borrow them for the duration of the
 *     (asynchronous) call on the given CUDA stream; nothing is allocated inside kb_step.
 *   - there is no CPU fallback: kb_create fails with KB_ERR_NO_DEVICE without an sm_100 GPU.
 */
#ifndef KB_B200_H
#define KB_B200_H

#ifndef __CUDACC_RTC__   /* the library's run-time compiled step kernel includes this header too */
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define KB_ABI_VERSION 1

#define KB_MAX_POLY_VERTS 8   /* b2_maxPolygonVertices (Box2D default) */
#define KB_MAX_FIXTURES 3     /* CForm has 3 sub-polygons (lib/body.py:327-329) */
#define KB_MAX_LIGHTS 4       /* children of a CompositeLight (lib/light.py:99-148) */
#define KB_BODY_STATE_FLOATS 12

typedef enum KbError {
  KB_OK = 0,
  KB_ERR_INVALID = -1,      /* bad argument / scene description */
  KB_ERR_NO_DEVICE = -2,    /* no sm_100 CUDA device: there is no CPU fallback */
  KB_ERR_CUDA = -3,         /* CUDA runtime error, see kb_last_error() */
  KB_ERR_CAPACITY = -4,     /* scene exceeds compiled / shared-memory capacity */
  KB_ERR_UNSUPPORTED = -5
} KbError;

/* shape of one fixture (lib/body.py:136-142 box, :187-192 circle, :245-251 polygon) */
typedef enum KbShape { KB_SHAPE_CIRCLE = 0, KB_SHAPE_POLYGON = 1, KB_SHAPE_BOX = 2 } KbShape;

/* controller attached to a body (lib/kilobot.py) */
typedef enum KbBodyKind {
  KB_BODY_OBJECT = 0,                 /* pushable object, no controller (lib/body.py) */
  KB_KILOBOT_PHOTOTAXIS = 1,          /* PhototaxisKilobot      lib/kilobot.py:303-333 + :86-127 */
  KB_KILOBOT_SIMPLE_PHOTOTAXIS = 2,   /* SimplePhototaxisKilobot lib/kilobot.py:171-203 */
  KB_KILOBOT_VELOCITY = 3,            /* SimpleVelocityControlKilobot lib/kilobot.py:213-258 */
  KB_KILOBOT_ACCELERATION = 4         /* SimpleAccelerationControlKilobot lib/kilobot.py:266-300 */
} KbBodyKind;

typedef enum KbLightType {
  KB_LIGHT_CIRCULAR = 1,   /* CircularGradientLight lib/light.py:151-195 (step :59-75) */
  KB_LIGHT_MOMENTUM = 2,   /* MomentumLight lib/light.py:274-319 */
  KB_LIGHT_LINEAR = 3      /* GradientLight lib/light.py:218-271 (intended semantics, see DESIGN.md D1) */
} KbLightType;

typedef struct KbFixtureDef {
  int32_t shape;          /* KbShape */
  int32_t vertex_count;   /* KB_SHAPE_POLYGON: number of input vertices (3..8) */
  float radius;           /* KB_SHAPE_CIRCLE: radius, b2 units */
  float hx, hy;           /* KB_SHAPE_BOX: half extents, b2 units (SetAsBox) */
  float density, friction, restitution;
  float vx[KB_MAX_POLY_VERTS]; /* KB_SHAPE_POLYGON: input vertices as passed to b2PolygonShape(vertices=) */
  float vy[KB_MAX_POLY_VERTS];
} KbFixtureDef;

typedef struct KbBodyDef {
  int32_t kind;           /* KbBodyKind */
  int32_t num_fixtures;   /* 1..KB_MAX_FIXTURES, creation order */
  float linear_damping;   /* lib/body.py:15, lib/kilobot.py:29 */
  float angular_damping;  /* lib/body.py:16, lib/kilobot.py:30 */
  KbFixtureDef fixtures[KB_MAX_FIXTURES];
} KbBodyDef;

typedef struct KbLightDef {
  int32_t type;              /* KbLightType */
  int32_t relative_actions;  /* SinglePositionLight: lib/light.py:48,69-72 */
  double radius;             /* lib/light.py:152 */
  double bounds_lo[2], bounds_hi[2];   /* position bounds (lib/light.py:44-46,74-75); +-inf allowed */
  double action_lo[2], action_hi[2];   /* action clip (lib/light.py:49-54,65-67) */
  double max_velocity;       /* MomentumLight lib/light.py:289-292,310-311; inf = unlimited */
} KbLightDef;

/* One scene = what KilobotsEnv._configure_environment builds (kilobots_env.py:111-113), minus poses. */
typedef struct KbSceneDesc {
  int32_t num_bodies;        /* objects first, then kilobots == Box2D creation order */
  int32_t num_objects;
  const KbBodyDef* bodies;   /* [num_bodies] */
  int32_t num_lights;        /* 0 = no light; >1 = CompositeLight over the children */
  const KbLightDef* lights;  /* [num_lights] */
  /* static table: b2ChainShape around the arena, kilobots_env.py:46-51 (b2 units) */
  float wall_x0, wall_y0, wall_x1, wall_y1;
  int32_t wall_edges;        /* 3 = open chain (pybox2d `vertices=`), 4 = closed loop, 0 = no table */
  float wall_friction;       /* b2FixtureDef default 0.2 */
  /* simulation constants, kilobots_env.py:25-28 */
  int32_t steps_per_action;  /* 10 */
  int32_t velocity_iterations, position_iterations; /* 10, 10 */
  float dt;                  /* 0.1 */
  /* Box2D-version switches (SURVEY Appendix B.9) */
  int32_t damping_mode;      /* 0 = Pade v/(1+h*c) (>=2.3.1), 1 = clamp(1-h*c,0,1) (<=2.3.0) */
  int32_t enable_toi;        /* b2World continuousPhysics (default true in Box2D) */
  int32_t enable_sleep;      /* b2World(doSleep=True) kilobots_env.py:45 */
  /* reward hook (kilobots_env.py:123-125): in-tree values are constants
     (yaml_kilobots_env.py:368-369 -> 0.0, kilobots_test_envs.py:89-91 -> 1.0) */
  float reward_const;
} KbSceneDesc;

typedef struct KbHandle KbHandle;

/* derived sizes of a created batch.  num_objects / num_kilobots are the largest counts over the scenes (Mmax, Nmax),
   num_bodies = Mmax + Nmax: every array shaped by the counts uses these maxima (see kb_create, padded body layout) */
typedef struct KbDims {
  int32_t num_envs, num_bodies, num_objects, num_kilobots;
  int32_t num_proxies;       /* max over scenes, wall edges included (they come first) */
  int32_t max_contacts;      /* per-env capacity of the persistent contact list */
  int32_t light_state_dim;   /* L: 2 per circular, 4 per momentum, 1 per linear light */
  int32_t action_dim;        /* A: 2 per circular/momentum, 1 per linear light */
  int32_t state_bytes_per_env;
} KbDims;

/* Per-env status bits written by kb_step / kb_reset */
#define KB_STATUS_CONTACT_OVERFLOW 1   /* persistent contact list hit max_contacts: pairs dropped */
#define KB_STATUS_NONFINITE 2          /* a pose became NaN/inf */
#define KB_STATUS_SOLVER_OVERFLOW 4    /* touching contacts exceeded the per-step solver capacity */

/* per-env counters (roofline accounting, SURVEY 8d); accumulated since the last reset */
#define KB_NUM_COUNTERS 8
#define KB_CNT_SUBSTEPS 0
#define KB_CNT_CONTACTS 1        /* sum over sub-steps of persistent contacts at sub-step start */
#define KB_CNT_POINTS 2          /* sum of manifold points fed to the solver */
#define KB_CNT_LEVELS 3          /* sum of Gauss-Seidel dependency levels */
#define KB_CNT_POS_ITERS 4       /* sum over islands of executed position iterations */
#define KB_CNT_TOI_EVENTS 5
#define KB_CNT_PAIR_TESTS 6
#define KB_CNT_ISLANDS 7

/* action routing of kb_step */
#define KB_ACTION_NONE 0     /* action=None: lights frozen (kilobots_env.py:171) */
#define KB_ACTION_LIGHT 1    /* action[E,A] drives the light(s) (kilobots_env.py:171-172) */
#define KB_ACTION_KILOBOTS 2 /* action[E,N,2] -> Kilobot.set_action (direct_control_kilobots_env.py:18-29) */

/*
 * Create a batch of num_envs environments.  scenes[num_scenes] are the distinct scene templates,
 * env_scene[num_envs] (host, may be NULL = all scene 0) picks one per env.  All scenes must agree in their lights,
 * light state / action dimensions and simulation constants; fixtures and the numbers of objects and kilobots may differ.
 * Padded body layout: with Mmax / Nmax the largest object / kilobot counts over the scenes, an env whose scene has M_e
 * objects and N_e kilobots keeps its objects at body indices 0..M_e-1 and its kilobots at Mmax..Mmax+N_e-1; the other
 * indices below Bmax = Mmax + Nmax are ABSENT bodies.  Body kinds must agree at every padded index two scenes both
 * populate.  Proxy ids are those of a compact world of the env's own bodies (table edges, then the fixtures of the
 * present bodies in body order): an absent body owns no proxy, is never awake and never moves.  Every array shaped by
 * the counts (poses, kb_velocity, observations, per-kilobot actions, the flat observation) uses the maxima; the pose
 * and action rows of absent bodies are ignored (they may hold anything, NaN included), their observation rows are quiet
 * NaN, kb_get_bodies reports them in the canonical state (all zero, xf.q.c = 1) and kb_get_mass_data as zeros.  More
 * than 62 bodies (Bmax) select the large-swarm tier, whose scenes must all be kilobots only.
 * max_contacts > 0: capacity of the persistent contact list per env; 0: the throughput default (8B + 32 pairs,
 * 3B + 9 touching contacts per solve -- ample for separated swarms; overflow sets KB_STATUS_* bits); < 0: one
 * slot for every proxy pair, so that no pair is ever dropped (the E = 1 drop-in facade: the reference's clipped
 * Gaussian spawn, yaml_kilobots_env.py:346-352, may stack kilobots on top of each other).  device = CUDA ordinal.
 */
int kb_create(const KbSceneDesc* scenes, int32_t num_scenes, const int32_t* env_scene,
              int32_t num_envs, int32_t max_contacts, int32_t device, KbHandle** out);
int kb_destroy(KbHandle* h);
int kb_get_dims(const KbHandle* h, KbDims* dims);
const char* kb_last_error(void);

/*
 * reset (kilobots_env.py:150-159): rebuild every env's bodies at the given poses with zero
 * velocity and fresh controllers, then run ONE world step without controllers (:157, :217-219).
 *   mask        device u8[E] or NULL (= all): which envs to reset
 *   body_pose   device f64[E,B,3]  (x m, y m, theta rad) -- Body.__init__ position/orientation (padded layout:
 *                                  rows of absent bodies are ignored)
 *   light_state device f64[E,L]    light position (+velocity / angle), may be NULL if no light
 *   kb_velocity device f64[E,N,2]  initial (v, omega) of velocity/acceleration-control kilobots
 *                                  (lib/kilobot.py:225-229); NULL = zeros
 */
int kb_reset(KbHandle* h, const uint8_t* mask, const double* body_pose, const double* light_state,
             const double* kb_velocity, void* stream);

/*
 * Reset with on-device scene sampling.  The reference re-draws its scene in every reset():
 * YamlKilobotsEnv._configure_environment (yaml_kilobots_env.py:194-198 objects, :256-283 lights, :299 shuffle of the
 * composite light's components, :327-354 kilobots) with numpy's global generator, one env at a time.  Here the reset
 * kernel draws the scene itself, as a pure function of (seed, global env id = env_id_base + env, episode count of the
 * env) -- Philox4x32-10, one block per draw -- so an auto-reset is ONE launch, never touches the host, and 1 GPU and
 * 8 GPUs reset an environment identically.  gym_kilobots_b200/sampler.py evaluates the same function in numpy.
 *   objects[i].mode   KB_SAMPLE_FIXED (pose) | KB_SAMPLE_RANDOM ((U^2 * size + lo) * 0.7, U * 2 pi - pi)
 *   lights[c].mode    per light component in the configuration's order: FIXED (init) | RANDOM (U^2 * size + lo) |
 *                     AT_OBJECT (radius 1.2 * extent / 2 around a random object); momentum lights start with speed .01
 *   shuffle_lights    composite light with init 'random': Fisher-Yates over the components.  Every permutation must be
 *                     a scene template of the batch (light constants are per scene); perm_scene[rank] = its scene index,
 *                     rank = lexicographic rank of (component at position 0, 1, ...).  The env's scene is switched.
 *   kilobot_mean_mode KB_SAMPLE_FIXED (kilobot_mean) | KB_SAMPLE_MEAN_LIGHT | KB_SAMPLE_MEAN_RANDOM
 */
#define KB_SAMPLE_FIXED 0
#define KB_SAMPLE_RANDOM 1
#define KB_SAMPLE_AT_OBJECT 2
#define KB_SAMPLE_MEAN_LIGHT 1
#define KB_SAMPLE_MEAN_RANDOM 2
typedef struct KbSampleObject {
  int32_t mode, reserved;
  double pose[3];      /* x m, y m, theta (KB_SAMPLE_FIXED) */
  double extent;       /* max(width, height) of the object as Body.width / Body.height report it */
} KbSampleObject;
typedef struct KbSampleLight {
  int32_t mode, reserved;
  double init[2];      /* position (KB_SAMPLE_FIXED); init[0] = angle of a linear light */
} KbSampleLight;
typedef struct KbSampleSpec {
  uint64_t seed;
  int64_t env_id_base;             /* global id of this handle's env 0 (rank * envs per rank) */
  double world_width, world_height;
  int32_t num_objects, num_lights;
  const KbSampleObject* objects;
  const KbSampleLight* lights;
  int32_t shuffle_lights, kilobot_mean_mode;
  const int32_t* perm_scene;       /* [num_lights!] or NULL */
  double kilobot_mean[2], kilobot_std;
} KbSampleSpec;
/* also restarts the episode counts; KB_ERR_UNSUPPORTED for a batch whose scenes differ in their object / kilobot counts
   (kb_set_sampler_mix draws such a batch).  Without shuffle_lights the env keeps its scene and perm_scene is not read. */
int kb_set_sampler(KbHandle* h, const KbSampleSpec* spec);
/*
 * On-device scene sampling for a batch that mixes K configurations (K = 1 is kb_set_sampler's case, without its refusal
 * of a mixed batch).  Every configuration c has its own spec; its scenes are specs[c].perm_scene: the scene of every
 * permutation (num_lights! entries with shuffle_lights, else 1 entry, the configuration's scene).  perm_scene is required
 * when K > 1; with K = 1 and no shuffle it is not read and the env keeps its scene, as with kb_set_sampler.  Every scene of
 * the batch belongs to at most one configuration, and every env's current scene to exactly one.  A spec's num_objects
 * equals the object count of each of its scenes, and its scenes have one kilobot count.
 *   weights  host f64[K] or NULL.  NULL: a sampled reset draws the configuration of the env's scene (kb_set_env_scene
 *            moves an env to another one).  Non-NULL (finite, >= 0, positive sum): every sampled reset first draws the
 *            configuration, c = first k with u < cdf[k] (cdf = the normalised cumulative weights, its last entry 1.0);
 *            u is a Philox uniform of its own stream keyed by (seed, global env id, episode).
 * Then the reset draws the scene of c exactly as kb_set_sampler would for a batch of c alone, in the padded body layout:
 * objects at 0..M_e-1, kilobots at Mmax + k; the rows of absent bodies in kb_get_sampled's body_pose are quiet NaN.
 * seed and env_id_base come from specs[0] and must agree over the specs.  Restarts the episode counts.  While such a
 * sampler is attached, kb_set_env_scene refuses a scene that belongs to no configuration.
 */
#define KB_SAMPLE_MAX_CONFIGS 16
int kb_set_sampler_mix(KbHandle* h, const KbSampleSpec* specs, int32_t num_specs, const double* weights);
/* device i32[E]: the scene each env was last reset with, written on `stream` without synchronising */
int kb_current_scenes(KbHandle* h, int32_t* out_device, void* stream);
/* like kb_reset, with the poses / light states drawn on the device; mask: device u8[E] or NULL */
int kb_reset_sampled(KbHandle* h, const uint8_t* mask, void* stream);
/* what the last sampled resets drew: host f64[E,B,3], f64[E,L], i32[E] scene per env, u32[E] resets so far (any may be NULL) */
int kb_get_sampled(KbHandle* h, double* body_pose, double* light_state, int32_t* env_scene, uint32_t* episodes);
/* overwrite the env -> scene map (host i32[E]); takes effect at the env's next reset (which may change the env's
   object / kilobot counts: see kb_get_body_counts) */
int kb_set_env_scene(KbHandle* h, const int32_t* env_scene);

/*
 * step (kilobots_env.py:161-215): steps_per_action sub-steps of
 *   light.step -> sensing -> controllers -> b2World.Step(dt, vel_iters, pos_iters)
 * then gathers the observation (get_state :115-118).  All pointers are device pointers.
 *   action        f64[E,A] (KB_ACTION_LIGHT) / f64[E,N,2] (KB_ACTION_KILOBOTS) / NULL
 *   obs_kilobots  f32[E,N,3]  (x m, y m, theta) = Body.get_pose (lib/body.py:63-65); absent kilobots: quiet NaN rows
 *   obs_objects   f32[E,M,3]  absent objects: quiet NaN rows
 *   obs_light     f64[E,L]    light.get_state()
 *   reward f32[E], done u8[E], status i32[E]; any output pointer may be NULL.
 */
int kb_step(KbHandle* h, const double* action, int32_t action_mode, float* obs_kilobots,
            float* obs_objects, double* obs_light, float* reward, uint8_t* done, int32_t* status,
            void* stream);

/*
 * Same call with HOST buffers (pinned or pageable): copies the action host->device, steps, and
 * copies the outputs device->host on `stream`, then synchronises the stream.  This is the call
 * the E=1 KilobotsEnv facade and the end-to-end benchmark use.
 */
int kb_step_host(KbHandle* h, const double* action, int32_t action_mode, float* obs_kilobots,
                 float* obs_objects, double* obs_light, float* reward, uint8_t* done,
                 int32_t* status, void* stream);

/* --- introspection for parity tests / checkpointing (host pointers; these synchronise) --- */
/* raw body state f32[E,B,12]: c.x c.y a v.x v.y w sleepTime awake xf.p.x xf.p.y xf.q.s xf.q.c (b2 units) */
int kb_get_bodies(KbHandle* h, float* out);
/* overwrite poses like Body.set_pose (lib/body.py:67-69 -> b2Body::SetTransform): f64[E,B,3] SI units */
int kb_set_poses(KbHandle* h, const double* body_pose);
/* the same for the bodies whose flag in body_mask (host u8[E,B], NULL = all) is set: Body.set_pose transforms ONE
   body and leaves every other body's sweep and proxies alone */
int kb_set_poses_masked(KbHandle* h, const double* body_pose, const uint8_t* body_mask);
/* per-env status word (KB_STATUS_* bits, sticky until the env is reset): host i32[E].  Also set by kb_reset's
   settle step, which kb_step's status output does not cover */
int kb_get_status(KbHandle* h, int32_t* out);
/* objects / kilobots of the scene each env was last reset with (before its first reset: its scene at kb_create):
   host i32[E] each, either may be NULL.  Object j < objects[e] is body j, kilobot k < kilobots[e] is body Mmax + k. */
int kb_get_body_counts(KbHandle* h, int32_t* objects, int32_t* kilobots);
/* persistent contact list in Box2D world-list order (newest first):
   pairs i32[E,max_contacts,4] = (proxyA, proxyB, touching, pointCount), count i32[E] */
int kb_get_contacts(KbHandle* h, int32_t* pairs, int32_t* count);
/* manifold impulses f32[E,max_contacts,4] = (n0, t0, n1, t1) in the same order */
int kb_get_impulses(KbHandle* h, float* out);
int kb_get_counters(KbHandle* h, uint64_t* out /* [E,KB_NUM_COUNTERS] */);
/* fat AABBs f32[E,P,4] (lower.x lower.y upper.x upper.y), wall edges first */
int kb_get_proxies(KbHandle* h, float* out);
/* controller state f64[E,N,4] + light state f64[E,L] */
int kb_get_controllers(KbHandle* h, double* ctrl, double* light);
/* full per-env state blob (checkpoint / bit-exact resume): state_bytes_per_env * E bytes */
int kb_get_state(KbHandle* h, void* out);
int kb_set_state(KbHandle* h, const void* in);
/* kb_step_host moves its six outputs with ONE device->host copy if the caller's buffers form one block laid out
   like the library's staging area: byte offsets of (obs_kilobots, obs_objects, obs_light, reward, status, done)
   from the start of that block, and its total size.  Any other arrangement of buffers works too (six copies). */
int kb_get_host_layout(const KbHandle* h, int64_t offsets[6], int64_t* total_bytes);
/* launch geometry of kb_step for this batch (reporting only): lanes of a warp that cooperate on one env
   (4, 8, 16 or 32), threads per block, blocks in the grid, dynamic shared memory per block in bytes */
typedef struct KbLaunchConfig {
  int32_t lanes_per_env, block_threads, grid_blocks, smem_bytes_per_block;
  int32_t state_words_per_env;   /* 32-bit words of per-env state resident in shared memory during a launch */
  int32_t smem_words_per_env;    /* state + solver scratch */
  /* the lane-group step kernel compiled at kb_create for this batch's layout (offsets, counts and solver constants as
   * immediates; same results as the generic kernel): 1 when it runs, 0 when the generic kb_step_kernel<LPE> runs.
   * KB_JIT=0 asks for the generic kernel, KB_JIT=1 makes kb_create fail when the specialised one cannot be had;
   * compiled kernels are cached under $KB_JIT_CACHE (default ~/.cache/gym_kilobots_b200). */
  int32_t specialised;
  float jit_ms;                  /* its compile time in kb_create, ms (0: taken from a cache) */
  char jit_reason[256];          /* why the generic kernel runs ("" when specialised) */
} KbLaunchConfig;
int kb_get_launch_config(const KbHandle* h, KbLaunchConfig* cfg);
/* Needs no GPU: the source kb_create generates for the specialised step kernel of a lane-group batch of `scenes`
 * (the batch's layout as constants; the kernel's headers are embedded in the library) into source[source_cap].  With
 * compile != 0 it also compiles it with NVRTC (no cache, nothing loaded) and writes NVRTC's log, ptxas's resource
 * report included, into log[log_cap] and the compile time into *compile_ms.  KB_ERR_INVALID for a large-swarm batch. */
int kb_jit_step_source(const KbSceneDesc* scenes, int32_t num_scenes, int32_t max_contacts, int32_t compile,
                       char* source, int64_t source_cap, char* log, int64_t log_cap, double* compile_ms);
/* derived mass data per scene: f32[num_scenes,B,4] = invMass invI localCenter.x localCenter.y */
int kb_get_mass_data(KbHandle* h, float* out);

/* ---------------------------------------------------------------------------------------------
 * Task layer -- an EXTENSION beyond the reference (SURVEY.md 8(a) row a13 and 8(f) rows n1, n3).
 * The reference's get_reward / has_finished / get_info (kilobots_env.py:123-131) are abstract hooks whose
 * in-tree implementations return constants (KB_TASK_CONST below, the default: reward = reward_const,
 * done = 0).  The other modes evaluate a task reward, the termination flag and episode statistics inside
 * kb_step's gather, and can emit the flat observation that YamlKilobotsEnv.observation_space describes
 * (yaml_kilobots_env.py:163-178: kilobots (x, y) * N, light state, objects (x, y, sin theta, cos theta) * M),
 * so that a training loop never leaves the device.  All task arithmetic is float64.
 *   error before / after the env-step:  d = |subject - target| (m), a = |wrap(theta - target_theta)| (rad)
 *   subject = pose of object `object` (KB_TASK_OBJECT_TO_TARGET; every scene must have it) or the mean position of
 *             the env's own kilobots (KB_TASK_SWARM_TO_TARGET, a = 0)
 *   reward  = w_position * (d0 - d1) + w_orientation * (a0 - a1) - step_penalty + (success ? success_bonus : 0)
 *   success = d1 <= position_tolerance && a1 <= orientation_tolerance
 *   done    = success || (max_episode_steps > 0 && episode length >= max_episode_steps)
 * kb_reset zeroes the episode return / length of the envs it resets. */
#define KB_TASK_CONST 0
#define KB_TASK_OBJECT_TO_TARGET 1
#define KB_TASK_SWARM_TO_TARGET 2
typedef struct KbTaskDef {
  int32_t mode;               /* KB_TASK_* */
  int32_t object;             /* object index (KB_TASK_OBJECT_TO_TARGET) */
  int32_t max_episode_steps;  /* time limit in env-steps, 0 = none */
  int32_t reserved;
  double w_position, w_orientation, step_penalty, success_bonus;
  double position_tolerance, orientation_tolerance;
} KbTaskDef;
/* per-env episode statistics, f64[E,KB_EPISODE_STATS] */
#define KB_EPISODE_STATS 6
#define KB_EP_RETURN 0        /* sum of rewards since the last reset */
#define KB_EP_LENGTH 1        /* env-steps since the last reset */
#define KB_EP_POSITION_ERROR 2
#define KB_EP_ORIENTATION_ERROR 3
#define KB_EP_SUCCESS 4       /* 1 if the last step met both tolerances */
#define KB_EP_DONE_COUNT 5    /* number of env-steps that returned done since kb_set_task */
/* target: host f64[E,3] = (x m, y m, theta rad) per env; NULL keeps the current targets (zeros initially) */
int kb_set_task(KbHandle* h, const KbTaskDef* task, const double* target);
int kb_get_episode_stats(KbHandle* h, double* out /* host f64[E,KB_EPISODE_STATS] */);
/* The rank-local half of "NCCL used only to all-reduce episode statistics" (BASELINE.json north_star; the reference's
   per-env hook is get_info, kilobots_env.py:130-131): sums over this handle's envs, written to a DEVICE buffer of
   KB_REDUCED_STATS doubles on `stream` (one block, fixed summation order), ready for ncclAllReduce(sum):
   [0] envs, [1..6] sums of the KB_EP_* statistics, [7] envs whose status word is non-zero. */
#define KB_REDUCED_STATS 8
int kb_reduce_episode_stats(KbHandle* h, double* out_device, void* stream);
/* device f32[E, 2N + L + 4M] written by every following kb_step (NULL unbinds); see kb_flat_observation_dim */
int kb_bind_flat_observation(KbHandle* h, float* obs_flat);
int kb_flat_observation_dim(const KbHandle* h);

/*
 * Per-kilobot local observations: what each kilobot would sense itself, in its own frame -- the input of a swarm policy
 * shared across the kilobots.  Computed from the state the handle holds after the last call on `stream` (kb_step*,
 * kb_reset*, kb_set_poses*, kb_set_state), for the env's present kilobots.  Output: device f32[E, Nmax, D]; row k of env e
 * belongs to padded kilobot k, the rows of absent kilobots are quiet NaN.  Per body b: p_b = the position kb_step reports
 * in obs_kilobots / obs_objects, (float)((double)xf.p / 25.0) in metres, and (s_b, c_b) = xf.q.  Float32 arithmetic, every
 * operation rounded separately.  The parts selected in `parts` follow each other in this order:
 *   KB_LOCAL_NEIGHBOURS  1 + 4K columns: n_i = the number of other present kilobots j of the env with d2 <= radius^2
 *                        (dx = p_j.x - p_i.x, dy = p_j.y - p_i.y, d2 = dx*dx + dy*dy; not capped at K), then K slots
 *                        ascending by (d2, j) of (c_i*dx + s_i*dy, -s_i*dx + c_i*dy, sqrtf(d2), 1); unfilled slots are 0.
 *   KB_LOCAL_OBJECTS     5 * Mmax columns: per object slot j the env has, its position in the kilobot's frame as above,
 *                        cos = c_j*c_i + s_j*s_i, sin = s_j*c_i - c_j*s_i, 1; zeros for a slot it does not have.
 *   KB_LOCAL_LIGHT       3 columns: the light value at the kilobot's light sensor (the point senseControl reads: the body
 *                        origin of a SimplePhototaxisKilobot, the rear point (0, -r) of the others) and its gradient rotated
 *                        into the body frame (c*gx + s*gy, -s*gx + c*gy), float64 with (double) of xf.q, then rounded to
 *                        float32.  Composite light: the sum of the values, the gradient of the brightest child.
 * max_neighbours (K) must be in 1..32, radius (metres) finite and > 0.  KB_LOCAL_FORCE_GRID=1 in the environment makes
 * every batch take the uniform-grid kernel of large swarms (same result).
 */
#define KB_LOCAL_NEIGHBOURS 1
#define KB_LOCAL_OBJECTS 2
#define KB_LOCAL_LIGHT 4
typedef struct KbLocalObsDef {
  float radius;
  int32_t max_neighbours;
  int32_t parts;   /* KB_LOCAL_* bits */
  int32_t pad;
} KbLocalObsDef;
/* D of the def on this batch, or a negative KbError */
int kb_local_observation_dim(const KbHandle* h, const KbLocalObsDef* def);
/* out: device f32[E, Nmax, D]; mask: device u8[E] or NULL = every env (rows of unmasked envs are not written).
   Asynchronous on `stream`: no allocation, no host synchronisation. */
int kb_local_observation(KbHandle* h, const KbLocalObsDef* def, const uint8_t* mask, float* out, void* stream);

/* Off-screen rasteriser (SURVEY.md 8(f) n4): the picture KilobotsEnv.render draws through
 * kb_rendering.KilobotsViewer (kilobots_env.py:221-275) -- table, objects, kilobots, light -- for num_images
 * environments, straight from the device state.  env_ids: host i32[num_images]; rgb: DEVICE u8[num_images,
 * height, width, 3], row 0 = top of the arena (y = +world_height / 2).  Asynchronous on `stream`. */
int kb_render(KbHandle* h, const int32_t* env_ids, int32_t num_images, int32_t width, int32_t height,
              uint8_t* rgb, void* stream);

/* Self-test of the kernels' arithmetic (no reference counterpart; see kb_sqrt_u / kb_rcp_u / kb_div_u in
 * csrc/kb_types.cuh): the straight-line square root and reciprocal are compared with sqrtf(x) and 1.0f / x on all 2^32
 * float bit patterns, the division with a / b on 2^(32 + div_rounds_log2) pseudo-random pairs (half of them with both
 * operands inside the fast path's exponent window); inputs the forms hand back to the plain operators are skipped.
 * mismatches: host u64[6] = differing results of (sqrt, reciprocal, division), the number of comparisons made, and
 * for the position solver's kilobot-kilobot step run the way the kernels run it (straight-line pass, rows stored, exact
 * pass out of line when a range test fired) against the plain operators on 2^26 pairs of bodies incl. degenerate ones:
 * differing rows / verdicts, and how many cases took the exact pass.  Bit-exact parity with Box2D's x86-64 arithmetic
 * needs entries 0, 1, 2 and 4 to be 0.  device < 0: the current device. */
int kb_selftest_exact_math(int32_t device, int32_t div_rounds_log2, uint64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* KB_B200_H */
