// CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED (see kbo_math.h).
// kbo_env.cpp -- the Python side of the reference's hot path restated in C++ (float64 where the
// reference uses numpy, float32 where values cross into Box2D), plus the kbo_* C entry points that
// mirror include/kb_b200.h with HOST pointers.
//   KilobotsEnv.step / reset / get_state      gym_kilobots/envs/kilobots_env.py:115-118,150-219
//   lights                                    gym_kilobots/lib/light.py:59-75,122-141,176-189,237-253,300-316
//   controllers                               gym_kilobots/lib/kilobot.py:54-61,86-127,188-203,235-258,283-300,318-333
//   body construction                         gym_kilobots/lib/body.py:18-38,129-142,181-192,217-251
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "../include/kb_b200.h"
#include "kbo_world.h"

namespace kbo {

struct LightState {
  double pos[2] = {0.0, 0.0};
  double vel[2] = {0.0, 0.0};
  double angle = 0.0;
};

struct KilobotCtrl {
  int kind = 0;
  int turnRight = 0;  // __turn_direction: 0 = 'left' (motors 255,0), 1 = 'right' (motors 0,255)
  double threshold = -std::numeric_limits<double>::infinity();
  int updateCounter = 0;
  int noChangeCounter = 0;
  double velocity[2] = {0.0, 0.0};      // SimpleVelocityControlKilobot._velocity
  double acceleration[2] = {0.0, 0.0};  // SimpleAccelerationControlKilobot._acceleration
  double lightValue = 0.0;
  double lightGrad[2] = {0.0, 0.0};
};

struct Scene {
  KbSceneDesc desc;
  std::vector<KbBodyDef> bodies;
  std::vector<KbLightDef> lights;
};

struct Env {
  World* world = nullptr;
  int scene = 0;
  std::vector<Body*> bodies;  // objects then kilobots
  std::vector<KilobotCtrl> ctrl;
  std::vector<LightState> lights;
  int status = 0;
  // task layer (extension, include/kb_b200.h "Task layer")
  double target[3] = {0.0, 0.0, 0.0};
  double stats[KB_EPISODE_STATS] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
};

struct Handle {
  std::vector<Scene> scenes;
  std::vector<Env> envs;
  int numBodies = 0, numObjects = 0, numKilobots = 0, numLights = 0;
  int lightStateDim = 0, actionDim = 0, maxContacts = 0, numProxies = 0;
  int threads = 1;
  KbTaskDef task = {};
  float* obsFlat = nullptr;
  // Kilobot.step single-motor constants (lib/kilobot.py:103-121), float32 b2Vec2 of translation*25
  float transRight[2], transLeft[2];
  float omegaRight, omegaLeft;
};

static thread_local std::string g_err;

static int LightStateDim(const KbLightDef& l) {
  return l.type == KB_LIGHT_MOMENTUM ? 4 : (l.type == KB_LIGHT_LINEAR ? 1 : 2);
}
static int LightActionDim(const KbLightDef& l) { return l.type == KB_LIGHT_LINEAR ? 1 : 2; }

static void ComputeMotorConstants(Handle* h, double dt) {
  // lib/kilobot.py:9-13,23
  const double radius = 0.0165;
  (void)radius;
  const double legLeft[2] = {-0.013, -0.009};
  const double legRight[2] = {+0.013, -0.009};
  const double maxAngular = 0.5 * M_PI;
  {  // motor_right branch :103-111 (uses _leg_left)
    double av = 255 / 255. * maxAngular;
    double ad = av * dt;
    double c = std::cos(ad), s = std::sin(ad);
    double tx = legLeft[0] - (c * legLeft[0] + (-s) * legLeft[1]);
    double ty = legLeft[1] - (s * legLeft[0] + c * legLeft[1]);
    h->transRight[0] = (float)(tx * 25.0);
    h->transRight[1] = (float)(ty * 25.0);
    h->omegaRight = (float)av;
  }
  {  // motor_left branch :113-121 (uses _leg_right)
    double av = -255 / 255. * maxAngular;
    double ad = av * dt;
    double c = std::cos(ad), s = std::sin(ad);
    double tx = legRight[0] - (c * legRight[0] + (-s) * legRight[1]);
    double ty = legRight[1] - (s * legRight[0] + c * legRight[1]);
    h->transLeft[0] = (float)(tx * 25.0);
    h->transLeft[1] = (float)(ty * 25.0);
    h->omegaLeft = (float)av;
  }
}

static Shape MakeShape(const KbFixtureDef& fd) {
  Shape s;
  if (fd.shape == KB_SHAPE_CIRCLE) {
    s.type = kCircle;
    s.radius = fd.radius;
    s.p.SetZero();
  } else if (fd.shape == KB_SHAPE_BOX) {
    s.SetAsBox(fd.hx, fd.hy);
  } else {
    Vec2 v[KB_MAX_POLY_VERTS];
    for (int i = 0; i < fd.vertex_count; ++i) v[i].Set(fd.vx[i], fd.vy[i]);
    s.SetPolygon(v, fd.vertex_count);
  }
  return s;
}

// KilobotsEnv.reset (kilobots_env.py:150-159) for one env: fresh world (canonical proxy ids,
// SURVEY B.7), table, objects, kilobots, then ONE world step without controllers.
static void ResetEnv(Handle* h, Env* e, const double* pose /*[B,3]*/, const double* light /*[L]*/,
                     const double* kbVel /*[N,2] or null*/) {
  const Scene& sc = h->scenes[e->scene];
  delete e->world;
  e->world = new World();
  World* w = e->world;
  w->dampingMode = sc.desc.damping_mode;
  w->continuousPhysics = sc.desc.enable_toi != 0;
  w->allowSleep = sc.desc.enable_sleep != 0;
  w->CreateTable(sc.desc.wall_x0, sc.desc.wall_y0, sc.desc.wall_x1, sc.desc.wall_y1, sc.desc.wall_edges,
                 sc.desc.wall_friction);
  e->bodies.clear();
  e->ctrl.assign(h->numKilobots, KilobotCtrl());
  e->status = 0;
  for (int b = 0; b < h->numBodies; ++b) {
    const KbBodyDef& bd = sc.bodies[b];
    // lib/body.py:33: b2Vec2(*(_world_scale * position)) -- float64 multiply, then float32
    float px = (float)(25.0 * pose[3 * b + 0]);
    float py = (float)(25.0 * pose[3 * b + 1]);
    float ang = (float)pose[3 * b + 2];
    Body* body = w->CreateBody(px, py, ang, bd.linear_damping, bd.angular_damping);
    for (int f = 0; f < bd.num_fixtures; ++f) {
      const KbFixtureDef& fd = bd.fixtures[f];
      w->CreateFixture(body, MakeShape(fd), fd.density, fd.friction, fd.restitution);
    }
    e->bodies.push_back(body);
    if (b >= h->numObjects) {
      KilobotCtrl& kc = e->ctrl[b - h->numObjects];
      kc.kind = bd.kind;
      if (kbVel && (bd.kind == KB_KILOBOT_VELOCITY || bd.kind == KB_KILOBOT_ACCELERATION)) {
        kc.velocity[0] = kbVel[2 * (b - h->numObjects) + 0];
        kc.velocity[1] = kbVel[2 * (b - h->numObjects) + 1];
      }
    }
  }
  e->lights.assign(h->numLights, LightState());
  int off = 0;
  for (int l = 0; l < h->numLights; ++l) {
    const KbLightDef& ld = sc.lights[l];
    LightState& ls = e->lights[l];
    if (ld.type == KB_LIGHT_LINEAR) {
      ls.angle = light[off];
    } else {
      ls.pos[0] = light[off];
      ls.pos[1] = light[off + 1];
      if (ld.type == KB_LIGHT_MOMENTUM) {
        ls.vel[0] = light[off + 2];
        ls.vel[1] = light[off + 3];
      }
    }
    off += LightStateDim(ld);
  }
  w->Step(sc.desc.dt, sc.desc.velocity_iterations, sc.desc.position_iterations);  // :157
}

static inline double ClipD(double a, double lo, double hi) {
  // np.minimum(np.maximum(a, lo), hi)
  double m = a > lo ? a : lo;
  return m < hi ? m : hi;
}

// light.step (lib/light.py)
static void LightStep(const KbLightDef& ld, LightState* ls, const double* action, double dt) {
  if (ld.type == KB_LIGHT_CIRCULAR) {  // SinglePositionLight.step :59-75
    double a0 = ClipD(action[0], ld.action_lo[0], ld.action_hi[0]);
    double a1 = ClipD(action[1], ld.action_lo[1], ld.action_hi[1]);
    if (ld.relative_actions) {
      ls->pos[0] += a0 * dt;
      ls->pos[1] += a1 * dt;
    } else {
      ls->pos[0] = a0;
      ls->pos[1] = a1;
    }
    ls->pos[0] = ClipD(ls->pos[0], ld.bounds_lo[0], ld.bounds_hi[0]);
    ls->pos[1] = ClipD(ls->pos[1], ld.bounds_lo[1], ld.bounds_hi[1]);
  } else if (ld.type == KB_LIGHT_MOMENTUM) {  // MomentumLight.step :300-316
    double a0 = ClipD(action[0], ld.action_lo[0], ld.action_hi[0]);
    double a1 = ClipD(action[1], ld.action_lo[1], ld.action_hi[1]);
    ls->vel[0] += a0 * dt;
    ls->vel[1] += a1 * dt;
    double n = std::sqrt(ls->vel[0] * ls->vel[0] + ls->vel[1] * ls->vel[1]);
    if (n > ld.max_velocity) {
      double f = ld.max_velocity / n;
      ls->vel[0] *= f;
      ls->vel[1] *= f;
    }
    ls->pos[0] += ls->vel[0] * dt;
    ls->pos[1] += ls->vel[1] * dt;
    ls->pos[0] = ClipD(ls->pos[0], ld.bounds_lo[0], ld.bounds_hi[0]);
    ls->pos[1] = ClipD(ls->pos[1], ld.bounds_lo[1], ld.bounds_hi[1]);
  } else {  // GradientLight.step :237-253 (absolute angle action)
    double a = ClipD(action[0], ld.action_lo[0], ld.action_hi[0]);
    ls->angle = a;
    if (ls->angle < -M_PI) ls->angle += 2 * M_PI;
    if (ls->angle > M_PI) ls->angle -= 2 * M_PI;
  }
}

// value_and_gradients at one sensor position (lib/light.py:176-189; linear light: intended
// semantics value = pos . vec, gradient = vec -- DESIGN.md D1)
static void LightValueGrad(const KbLightDef& ld, const LightState& ls, double px, double py,
                           double* value, double* gx, double* gy) {
  if (ld.type == KB_LIGHT_LINEAR) {
    double vx, vy;  // np.cos/np.sin (lib/light.py:253) via the shared double sincos
    SinCosD(ls.angle, &vy, &vx);
    *value = vx * px + vy * py;
    *gx = vx;
    *gy = vy;
    return;
  }
  double g0 = -1 * (px - ls.pos[0]);
  double g1 = -1 * (py - ls.pos[1]);
  double norm = std::sqrt(g0 * g0 + g1 * g1);
  double v = 1.0;
  v -= norm / ld.radius;
  v = v < 1. ? v : 1.;
  v = v > .0 ? v : .0;
  v *= 255;
  if (norm == 0.0) {  // reference yields NaN here (0/0); guarded, DESIGN.md D3
    g0 = 0.0;
    g1 = 0.0;
  } else {
    g0 /= norm;
    g1 /= norm;
  }
  if (norm > ld.radius) {
    g0 *= .0;
    g1 *= .0;
  }
  *value = v;
  *gx = g0;
  *gy = g1;
}

// Kilobot.step for one kilobot (kilobots_env.py:183-184 -> lib/kilobot.py)
static void RunController(const Handle* h, KilobotCtrl& kc, Body* b, float dtf, double dt) {
  switch (kc.kind) {
    case KB_KILOBOT_PHOTOTAXIS: {
      // _loop lib/kilobot.py:318-333
      if (kc.updateCounter % 6) {
        kc.updateCounter += 1;
      } else {
        kc.updateCounter += 1;
        double m = kc.lightValue;  // get_ambientlight :57-61 (falsy -> 0)
        if (m > kc.threshold || kc.noChangeCounter >= 15) {
          kc.threshold = m + .01;
          kc.turnRight = kc.turnRight ? 0 : 1;  // switch_directions :67-71
          kc.noChangeCounter = 0;
        } else {
          kc.noChangeCounter += 1;
        }
      }
      // Kilobot.step single-motor branches :103-127
      const float* t = kc.turnRight ? h->transRight : h->transLeft;
      float w_ = kc.turnRight ? h->omegaRight : h->omegaLeft;
      Vec2 wv = b->GetWorldVector(Vec2(t[0], t[1]));
      // b2Vec2 / _world_scale / time_step, then * _world_scale: float32 ops in pybox2d
      Vec2 lv(wv.x / 25.0f, wv.y / 25.0f);
      lv.Set(lv.x / dtf, lv.y / dtf);
      lv.Set(lv.x * 25.0f, lv.y * 25.0f);
      b->SetAngularVelocity(w_);
      b->SetLinearVelocity(lv);
    } break;
    case KB_KILOBOT_SIMPLE_PHOTOTAXIS: {  // :191-203
      double mx = kc.lightGrad[0], my = kc.lightGrad[1];
      double n = std::sqrt(mx * mx + my * my);
      if (n > 0.01) {
        mx = mx / n * 0.01;
        my = my / n * 0.01;
      }
      mx *= 25.0;
      my *= 25.0;
      b->SetLinearVelocity(Vec2((float)mx, (float)my));
      b->linearDamping = .0f;
    } break;
    case KB_KILOBOT_ACCELERATION:  // :294-300
      kc.velocity[0] += kc.acceleration[0] * dt;
      kc.velocity[1] += kc.acceleration[1] * dt;
      kc.velocity[0] = kc.velocity[0] > .0 ? kc.velocity[0] : .0;
      kc.velocity[1] = kc.velocity[1] > -0.5 * M_PI ? kc.velocity[1] : -0.5 * M_PI;
      kc.velocity[0] = kc.velocity[0] < 0.01 ? kc.velocity[0] : 0.01;
      kc.velocity[1] = kc.velocity[1] < 0.5 * M_PI ? kc.velocity[1] : 0.5 * M_PI;
      // fallthrough
    case KB_KILOBOT_VELOCITY: {  // :253-258
      double ang = (double)b->sweep.a;
      double lx, ly;  // np.cos/np.sin via the shared double sincos (kbo_math.h)
      SinCosD(ang, &ly, &lx);
      lx *= kc.velocity[0] * 25.0;
      ly *= kc.velocity[0] * 25.0;
      b->SetLinearVelocity(Vec2((float)lx, (float)ly));
      b->SetAngularVelocity((float)kc.velocity[1]);
    } break;
    default: break;
  }

}

static void StepEnv(Handle* h, Env* e, const double* action, int actionMode) {
  const Scene& sc = h->scenes[e->scene];
  World* w = e->world;
  const int M = h->numObjects, N = h->numKilobots;
  const double dt = 1. / 10;  // KilobotsEnv.sim_step, kilobots_env.py:32 (float64 0.1)
  const float dtf = sc.desc.dt;

  if (actionMode == KB_ACTION_KILOBOTS) {  // direct_control_kilobots_env.py:18-29 -> set_action
    for (int k = 0; k < N; ++k) {
      KilobotCtrl& kc = e->ctrl[k];
      const double* a = action ? action + 2 * k : nullptr;
      if (kc.kind == KB_KILOBOT_VELOCITY) {  // lib/kilobot.py:235-241, action_space :216-218
        if (a) {
          kc.velocity[0] = ClipD(a[0], .0, 0.01) ;
          kc.velocity[1] = ClipD(a[1], -0.5 * M_PI, 0.5 * M_PI);
        } else {
          kc.velocity[0] = kc.velocity[1] = .0;
        }
      } else if (kc.kind == KB_KILOBOT_ACCELERATION) {  // :283-289, action_space :269
        if (a) {
          kc.acceleration[0] = ClipD(a[0], -.005, .005);
          kc.acceleration[1] = ClipD(a[1], -.2 * M_PI, .2 * M_PI);
        } else {
          kc.acceleration[0] = kc.acceleration[1] = .0;
        }
      }
    }
  }

  for (int step = 0; step < sc.desc.steps_per_action; ++step) {
    // light.step, kilobots_env.py:171-172 (CompositeLight.step lib/light.py:122-127)
    if (actionMode == KB_ACTION_LIGHT && action && h->numLights > 0) {
      int off = 0;
      for (int l = 0; l < h->numLights; ++l) {
        LightStep(sc.lights[l], &e->lights[l], action + off, dt);
        off += LightActionDim(sc.lights[l]);
      }
    }
    // sensing, kilobots_env.py:174-180
    if (h->numLights > 0) {
      for (int k = 0; k < N; ++k) {
        Body* b = e->bodies[M + k];
        KilobotCtrl& kc = e->ctrl[k];
        double sx, sy;
        if (kc.kind == KB_KILOBOT_SIMPLE_PHOTOTAXIS) {  // get_position lib/kilobot.py:188-189
          sx = (double)b->xf.p.x / 25.0;
          sy = (double)b->xf.p.y / 25.0;
        } else {  // get_world_point((0, -r)) lib/kilobot.py:54-55, lib/body.py:84-85
          Vec2 lp((float)(25.0 * 0.0), (float)(25.0 * -0.0165));
          Vec2 wp = b->GetWorldPoint(lp);
          sx = (double)wp.x / 25.0;
          sy = (double)wp.y / 25.0;
        }
        double value = 0.0, gx = 0.0, gy = 0.0;
        if (h->numLights == 1) {
          LightValueGrad(sc.lights[0], e->lights[0], sx, sy, &value, &gx, &gy);
        } else {  // CompositeLight.value_and_gradients lib/light.py:137-141
          double best = 0.0;
          for (int l = 0; l < h->numLights; ++l) {
            double v, g0, g1;
            LightValueGrad(sc.lights[l], e->lights[l], sx, sy, &v, &g0, &g1);
            value += v;
            if (l == 0 || v > best) {  // np.argmax: first maximum
              best = v;
              gx = g0;
              gy = g1;
            }
          }
        }
        kc.lightValue = value;
        kc.lightGrad[0] = gx;
        kc.lightGrad[1] = gy;
      }
    }
    // controllers, kilobots_env.py:183-184
    for (int k = 0; k < N; ++k) RunController(h, e->ctrl[k], e->bodies[M + k], dtf, dt);
    w->Step(dtf, sc.desc.velocity_iterations, sc.desc.position_iterations);  // :187
  }
  for (Body* b : e->bodies) {
    if (!std::isfinite(b->xf.p.x) || !std::isfinite(b->xf.p.y) || !std::isfinite(b->sweep.a))
      e->status |= KB_STATUS_NONFINITE;
  }
  if (w->contactCount > h->maxContacts) e->status |= KB_STATUS_CONTACT_OVERFLOW;
}

// task layer: distance (m) / |angle| (rad) of the task's subject to the env's target (include/kb_b200.h)
static void TaskError(const Handle* h, const Env* e, double* dist, double* ang) {
  const KbTaskDef& tk = h->task;
  double px, py, th = 0.0;
  if (tk.mode == KB_TASK_OBJECT_TO_TARGET) {
    const Body* b = e->bodies[tk.object];
    px = (double)b->xf.p.x / 25.0;
    py = (double)b->xf.p.y / 25.0;
    th = (double)b->sweep.a;
  } else {
    double sx = 0.0, sy = 0.0;
    for (int b = h->numObjects; b < h->numBodies; ++b) {
      sx += (double)e->bodies[b]->xf.p.x / 25.0;
      sy += (double)e->bodies[b]->xf.p.y / 25.0;
    }
    px = sx / (double)h->numKilobots;
    py = sy / (double)h->numKilobots;
  }
  const double dx = px - e->target[0], dy = py - e->target[1];
  *dist = std::sqrt(dx * dx + dy * dy);
  *ang = tk.mode == KB_TASK_OBJECT_TO_TARGET ? std::fabs(std::remainder(th - e->target[2], 6.283185307179586)) : 0.0;
}

template <class F>
static void ParallelFor(Handle* h, F f) {
  const int E = (int)h->envs.size();
  const int T = std::max(1, std::min(h->threads, E));
  if (T == 1) {
    for (int i = 0; i < E; ++i) f(i);
    return;
  }
  std::vector<std::thread> pool;
  for (int t = 0; t < T; ++t)
    pool.emplace_back([=] {
      for (int i = t; i < E; i += T) f(i);
    });
  for (auto& th : pool) th.join();
}

}  // namespace kbo

using namespace kbo;

extern "C" {

const char* kbo_last_error(void) { return g_err.c_str(); }

int kbo_create(const KbSceneDesc* scenes, int32_t num_scenes, const int32_t* env_scene, int32_t num_envs,
               int32_t max_contacts, int32_t device, KbHandle** out) {
  (void)device;
  if (!scenes || num_scenes < 1 || num_envs < 1 || !out) {
    g_err = "kbo_create: invalid arguments";
    return KB_ERR_INVALID;
  }
  Handle* h = new Handle();
  h->scenes.resize(num_scenes);
  for (int s = 0; s < num_scenes; ++s) {
    Scene& sc = h->scenes[s];
    sc.desc = scenes[s];
    sc.bodies.assign(scenes[s].bodies, scenes[s].bodies + scenes[s].num_bodies);
    sc.lights.assign(scenes[s].lights, scenes[s].lights + scenes[s].num_lights);
    sc.desc.bodies = sc.bodies.data();
    sc.desc.lights = sc.lights.data();
    if (s > 0 && (scenes[s].num_bodies != scenes[0].num_bodies || scenes[s].num_objects != scenes[0].num_objects ||
                  scenes[s].num_lights != scenes[0].num_lights)) {
      g_err = "kbo_create: scenes disagree in body/light counts";
      delete h;
      return KB_ERR_INVALID;
    }
  }
  h->numBodies = scenes[0].num_bodies;
  h->numObjects = scenes[0].num_objects;
  h->numKilobots = h->numBodies - h->numObjects;
  h->numLights = scenes[0].num_lights;
  for (int l = 0; l < h->numLights; ++l) {
    h->lightStateDim += LightStateDim(h->scenes[0].lights[l]);
    h->actionDim += LightActionDim(h->scenes[0].lights[l]);
  }
  int maxP = 0;
  for (const Scene& sc : h->scenes) {
    int p = sc.desc.wall_edges;
    for (const KbBodyDef& b : sc.bodies) p += b.num_fixtures;
    maxP = std::max(maxP, p);
  }
  h->numProxies = maxP;
  // same default and rounding as the product library (kb_create): min(P(P-1)/2, 8B+32), up to a multiple of 4
  // same capacity rule as kb_create: > 0 the caller's, 0 the throughput default, < 0 every proxy pair
  h->maxContacts = ((max_contacts > 0 ? max_contacts
                                      : (max_contacts < 0 ? std::max(maxP * (maxP - 1) / 2, 4)
                                                          : std::min(maxP * (maxP - 1) / 2, 8 * h->numBodies + 32))) + 3) & ~3;
  if (h->maxContacts > 65535) h->maxContacts = 65532;
  ComputeMotorConstants(h, 1. / 10);
  h->envs.resize(num_envs);
  for (int i = 0; i < num_envs; ++i) h->envs[i].scene = env_scene ? env_scene[i] : 0;
  *out = reinterpret_cast<KbHandle*>(h);
  return KB_OK;
}

int kbo_destroy(KbHandle* hh) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h) return KB_OK;
  for (Env& e : h->envs) delete e.world;
  delete h;
  return KB_OK;
}

int kbo_set_threads(KbHandle* hh, int32_t n) {
  reinterpret_cast<Handle*>(hh)->threads = n < 1 ? 1 : n;
  return KB_OK;
}

int kbo_get_dims(const KbHandle* hh, KbDims* d) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  d->num_envs = (int)h->envs.size();
  d->num_bodies = h->numBodies;
  d->num_objects = h->numObjects;
  d->num_kilobots = h->numKilobots;
  d->num_proxies = h->numProxies;
  d->max_contacts = h->maxContacts;
  d->light_state_dim = h->lightStateDim;
  d->action_dim = h->actionDim;
  d->state_bytes_per_env = 0;
  return KB_OK;
}

int kbo_reset(KbHandle* hh, const uint8_t* mask, const double* body_pose, const double* light_state,
              const double* kb_velocity, void* stream) {
  (void)stream;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int B = h->numBodies, L = h->lightStateDim, N = h->numKilobots;
  ParallelFor(h, [&](int i) {
    if (mask && !mask[i]) return;
    h->envs[i].stats[KB_EP_RETURN] = h->envs[i].stats[KB_EP_LENGTH] = h->envs[i].stats[KB_EP_SUCCESS] = 0.0;
    ResetEnv(h, &h->envs[i], body_pose + (size_t)i * B * 3, light_state ? light_state + (size_t)i * L : nullptr,
             kb_velocity ? kb_velocity + (size_t)i * N * 2 : nullptr);
  });
  return KB_OK;
}

int kbo_step(KbHandle* hh, const double* action, int32_t action_mode, float* obs_kilobots, float* obs_objects,
             double* obs_light, float* reward, uint8_t* done, int32_t* status, void* stream) {
  (void)stream;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int M = h->numObjects, N = h->numKilobots, L = h->lightStateDim;
  const int A = action_mode == KB_ACTION_KILOBOTS ? 2 * N : h->actionDim;
  ParallelFor(h, [&](int i) {
    Env* e = &h->envs[i];
    if (!e->world) return;
    double d0 = 0.0, a0 = 0.0;
    if (h->task.mode != KB_TASK_CONST) TaskError(h, e, &d0, &a0);
    StepEnv(h, e, action ? action + (size_t)i * A : nullptr, action ? action_mode : KB_ACTION_NONE);
    float* flat = h->obsFlat ? h->obsFlat + (size_t)i * (2 * N + L + 4 * M) : nullptr;
    // get_state, kilobots_env.py:115-118; Body.get_pose lib/body.py:63-65
    for (int b = 0; b < M + N; ++b) {
      const Body* body = e->bodies[b];
      float* o = b < M ? (obs_objects ? obs_objects + ((size_t)i * M + b) * 3 : nullptr)
                       : (obs_kilobots ? obs_kilobots + ((size_t)i * N + (b - M)) * 3 : nullptr);
      const float ox = (float)((double)body->xf.p.x / 25.0), oy = (float)((double)body->xf.p.y / 25.0);
      if (flat) {  // YamlKilobotsEnv.observation_space layout (yaml_kilobots_env.py:163-178)
        if (b < M) {
          float* f = flat + 2 * N + L + 4 * b;
          f[0] = ox; f[1] = oy; f[2] = body->xf.q.s; f[3] = body->xf.q.c;
        } else {
          flat[2 * (b - M)] = ox;
          flat[2 * (b - M) + 1] = oy;
        }
      }
      if (!o) continue;
      o[0] = ox;
      o[1] = oy;
      o[2] = body->sweep.a;
    }
    double lightBuf[16];
    if (obs_light || flat) {
      double* o = obs_light ? obs_light + (size_t)i * L : lightBuf;
      int off = 0;
      for (int l = 0; l < h->numLights; ++l) {
        const KbLightDef& ld = h->scenes[e->scene].lights[l];
        const LightState& ls = e->lights[l];
        if (ld.type == KB_LIGHT_LINEAR) {
          o[off] = ls.angle;
        } else {
          o[off] = ls.pos[0];
          o[off + 1] = ls.pos[1];
          if (ld.type == KB_LIGHT_MOMENTUM) {
            o[off + 2] = ls.vel[0];
            o[off + 3] = ls.vel[1];
          }
        }
        off += LightStateDim(ld);
      }
      if (flat)
        for (int k = 0; k < L; ++k) flat[2 * N + k] = (float)o[k];
    }
    float rew = h->scenes[e->scene].desc.reward_const;
    uint8_t dn = 0;
    if (h->task.mode != KB_TASK_CONST) {
      const KbTaskDef& tk = h->task;
      double d1, a1;
      TaskError(h, e, &d1, &a1);
      const bool success = d1 <= tk.position_tolerance && a1 <= tk.orientation_tolerance;
      double r = tk.w_position * (d0 - d1);
      r = r + tk.w_orientation * (a0 - a1);
      r = r - tk.step_penalty;
      if (success) r = r + tk.success_bonus;
      const double len = e->stats[KB_EP_LENGTH] + 1.0;
      dn = (success || (tk.max_episode_steps > 0 && len >= (double)tk.max_episode_steps)) ? 1 : 0;
      e->stats[KB_EP_RETURN] += r;
      e->stats[KB_EP_LENGTH] = len;
      e->stats[KB_EP_POSITION_ERROR] = d1;
      e->stats[KB_EP_ORIENTATION_ERROR] = a1;
      e->stats[KB_EP_SUCCESS] = success ? 1.0 : 0.0;
      if (dn) e->stats[KB_EP_DONE_COUNT] += 1.0;
      rew = (float)r;
    }
    if (reward) reward[i] = rew;
    if (done) done[i] = dn;
    if (status) status[i] = e->status;
  });
  return KB_OK;
}

int kbo_step_host(KbHandle* hh, const double* action, int32_t action_mode, float* obs_kilobots,
                  float* obs_objects, double* obs_light, float* reward, uint8_t* done, int32_t* status,
                  void* stream) {
  return kbo_step(hh, action, action_mode, obs_kilobots, obs_objects, obs_light, reward, done, status, stream);
}

int kbo_get_bodies(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int B = h->numBodies;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    const Env& e = h->envs[i];
    for (int b = 0; b < B; ++b) {
      const Body* body = e.bodies[b];
      float* o = out + (i * B + b) * KB_BODY_STATE_FLOATS;
      o[0] = body->sweep.c.x;
      o[1] = body->sweep.c.y;
      o[2] = body->sweep.a;
      o[3] = body->linearVelocity.x;
      o[4] = body->linearVelocity.y;
      o[5] = body->angularVelocity;
      o[6] = body->sleepTime;
      o[7] = body->IsAwake() ? 1.0f : 0.0f;
      o[8] = body->xf.p.x;
      o[9] = body->xf.p.y;
      o[10] = body->xf.q.s;
      o[11] = body->xf.q.c;
    }
  }
  return KB_OK;
}

int kbo_set_poses_masked(KbHandle* hh, const double* pose, const uint8_t* body_mask) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int B = h->numBodies;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    Env& e = h->envs[i];
    for (int b = 0; b < B; ++b) {
      if (body_mask && !body_mask[i * B + b]) continue;
      const double* p = pose + (i * B + b) * 3;
      // lib/body.py:54-61: position * _world_scale (float64) -> b2Vec2 (float32)
      e.world->SetTransform(e.bodies[b], (float)(p[0] * 25.0), (float)(p[1] * 25.0), (float)p[2]);
    }
  }
  return KB_OK;
}

int kbo_set_poses(KbHandle* hh, const double* pose) { return kbo_set_poses_masked(hh, pose, nullptr); }

// env -> scene map (takes effect at the env's next reset): mirrors kb_set_env_scene, so that tests can replay the
// scene switches of the device-side sampler
int kbo_set_env_scene(KbHandle* hh, const int32_t* env_scene) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  for (size_t i = 0; i < h->envs.size(); ++i) {
    if (env_scene[i] < 0 || env_scene[i] >= (int)h->scenes.size()) return KB_ERR_INVALID;
    h->envs[i].scene = env_scene[i];
  }
  return KB_OK;
}

int kbo_get_status(KbHandle* hh, int32_t* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  for (size_t i = 0; i < h->envs.size(); ++i) out[i] = h->envs[i].status;
  return KB_OK;
}

int kbo_get_contacts(KbHandle* hh, int32_t* pairs, int32_t* count) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int C = h->maxContacts;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    const Env& e = h->envs[i];
    int n = 0;
    for (Contact* c = e.world->contactList; c; c = c->next) {
      if (n < C) {
        int32_t* o = pairs + (i * C + n) * 4;
        o[0] = c->fixtureA->proxyId;
        o[1] = c->fixtureB->proxyId;
        o[2] = c->IsTouching() ? 1 : 0;
        o[3] = c->manifold.pointCount;
      }
      ++n;
    }
    count[i] = n;
  }
  return KB_OK;
}

int kbo_get_impulses(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int C = h->maxContacts;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    const Env& e = h->envs[i];
    int n = 0;
    for (Contact* c = e.world->contactList; c && n < C; c = c->next, ++n) {
      float* o = out + (i * C + n) * 4;
      for (int j = 0; j < 2; ++j) {
        bool live = j < c->manifold.pointCount;
        o[2 * j] = live ? c->manifold.points[j].normalImpulse : 0.0f;
        o[2 * j + 1] = live ? c->manifold.points[j].tangentImpulse : 0.0f;
      }
    }
  }
  return KB_OK;
}

int kbo_get_counters(KbHandle* hh, uint64_t* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  for (size_t i = 0; i < h->envs.size(); ++i) {
    const WorldCounters& c = h->envs[i].world->counters;
    uint64_t* o = out + i * KB_NUM_COUNTERS;
    o[KB_CNT_SUBSTEPS] = c.substeps;
    o[KB_CNT_CONTACTS] = c.contacts;
    o[KB_CNT_POINTS] = c.points;
    o[KB_CNT_LEVELS] = c.levels;
    o[KB_CNT_POS_ITERS] = c.posIters;
    o[KB_CNT_TOI_EVENTS] = c.toiEvents;
    o[KB_CNT_PAIR_TESTS] = c.pairTests;
    o[KB_CNT_ISLANDS] = c.islands;
  }
  return KB_OK;
}

int kbo_get_proxies(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int P = h->numProxies;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    const Env& e = h->envs[i];
    for (int p = 0; p < P; ++p) {
      float* o = out + (i * P + p) * 4;
      if (p < (int)e.world->proxies.size()) {
        const AABB& a = e.world->proxies[p]->fatAABB;
        o[0] = a.lowerBound.x;
        o[1] = a.lowerBound.y;
        o[2] = a.upperBound.x;
        o[3] = a.upperBound.y;
      } else {
        o[0] = o[1] = o[2] = o[3] = 0.0f;
      }
    }
  }
  return KB_OK;
}

int kbo_get_controllers(KbHandle* hh, double* ctrl, double* light) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  const int N = h->numKilobots, L = h->lightStateDim;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    const Env& e = h->envs[i];
    if (ctrl) {
      for (int k = 0; k < N; ++k) {
        const KilobotCtrl& kc = e.ctrl[k];
        double* o = ctrl + (i * N + k) * 4;
        if (kc.kind == KB_KILOBOT_PHOTOTAXIS) {
          o[0] = kc.threshold;
          o[1] = (double)kc.turnRight;
          o[2] = (double)kc.updateCounter;
          o[3] = (double)kc.noChangeCounter;
        } else {
          o[0] = kc.velocity[0];
          o[1] = kc.velocity[1];
          o[2] = kc.acceleration[0];
          o[3] = kc.acceleration[1];
        }
      }
    }
    if (light) {
      double* o = light + i * L;
      int off = 0;
      for (int l = 0; l < h->numLights; ++l) {
        const KbLightDef& ld = h->scenes[e.scene].lights[l];
        const LightState& ls = e.lights[l];
        if (ld.type == KB_LIGHT_LINEAR) {
          o[off] = ls.angle;
        } else {
          o[off] = ls.pos[0];
          o[off + 1] = ls.pos[1];
          if (ld.type == KB_LIGHT_MOMENTUM) {
            o[off + 2] = ls.vel[0];
            o[off + 3] = ls.vel[1];
          }
        }
        off += LightStateDim(ld);
      }
    }
  }
  return KB_OK;
}

int kbo_set_task(KbHandle* hh, const KbTaskDef* task, const double* target) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  if (!h || !task) return KB_ERR_INVALID;
  if (task->mode < KB_TASK_CONST || task->mode > KB_TASK_SWARM_TO_TARGET) return KB_ERR_INVALID;
  if (task->mode == KB_TASK_OBJECT_TO_TARGET && (task->object < 0 || task->object >= h->numObjects)) return KB_ERR_INVALID;
  h->task = *task;
  for (size_t i = 0; i < h->envs.size(); ++i) {
    Env& e = h->envs[i];
    if (target)
      for (int k = 0; k < 3; ++k) e.target[k] = target[i * 3 + k];
    for (int k = 0; k < KB_EPISODE_STATS; ++k) e.stats[k] = 0.0;
  }
  return KB_OK;
}

int kbo_get_episode_stats(KbHandle* hh, double* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  for (size_t i = 0; i < h->envs.size(); ++i)
    for (int k = 0; k < KB_EPISODE_STATS; ++k) out[i * KB_EPISODE_STATS + k] = h->envs[i].stats[k];
  return KB_OK;
}

int kbo_bind_flat_observation(KbHandle* hh, float* obs_flat) {
  reinterpret_cast<Handle*>(hh)->obsFlat = obs_flat;
  return KB_OK;
}

int kbo_flat_observation_dim(const KbHandle* hh) {
  const Handle* h = reinterpret_cast<const Handle*>(hh);
  return 2 * h->numKilobots + h->lightStateDim + 4 * h->numObjects;
}

// Off-screen rasteriser mirror (include/kb_b200.h kb_render): same float32 expressions, pixel by pixel, from the
// oracle's own objects.  Draw semantics: kilobots_env.py:221-275, lib/body.py:156-157,202-203,279-281,
// lib/kilobot.py:129-145,205-210, lib/light.py:95-96,194-195.  rgb is a HOST buffer here.
int kbo_render(KbHandle* hh, const int32_t* env_ids, int32_t num_images, int32_t width, int32_t height, uint8_t* rgb,
               void* stream) {
  (void)stream;
  Handle* h = reinterpret_cast<Handle*>(hh);
  const float S = 25.0f;
  for (int img = 0; img < num_images; ++img) {
    const Env* e = &h->envs[env_ids[img]];
    const Scene& sc = h->scenes[e->scene];
    const float x0 = sc.desc.wall_x0, y0 = sc.desc.wall_y0, x1 = sc.desc.wall_x1, y1 = sc.desc.wall_y1;
    for (int py = 0; py < height; ++py)
      for (int px = 0; px < width; ++px) {
        const float x = x0 + ((float)px + 0.5f) * ((x1 - x0) / (float)width);
        const float y = y1 - ((float)py + 0.5f) * ((y1 - y0) / (float)height);
        float c[3] = {255.0f, 255.0f, 255.0f};
        const float hbx = std::fmax(0.0015f * S, (x1 - x0) / (float)width);
        const float hby = std::fmax(0.0015f * S, (y1 - y0) / (float)height);
        if (x - x0 < hbx || x1 - x < hbx || y - y0 < hby || y1 - y < hby) c[0] = c[1] = c[2] = 0.0f;
        for (int b = 0; b < h->numObjects; ++b) {
          const Body* body = e->bodies[b];
          const float dx = x - body->xf.p.x, dy = y - body->xf.p.y;
          for (const Fixture* f : body->fixtures) {
            bool inside;
            if (f->shape.type == kCircle) {
              inside = dx * dx + dy * dy <= f->shape.radius * f->shape.radius;
            } else {
              const float lx = body->xf.q.c * dx + body->xf.q.s * dy, ly = -body->xf.q.s * dx + body->xf.q.c * dy;
              inside = true;
              for (int i = 0; i < f->shape.count; ++i)
                inside = inside && (f->shape.normals[i].x * (lx - f->shape.vertices[i].x) +
                                    f->shape.normals[i].y * (ly - f->shape.vertices[i].y) <= 0.0f);
            }
            if (inside) { c[0] = 93.0f; c[1] = 133.0f; c[2] = 195.0f; }
          }
        }
        for (int b = h->numObjects; b < h->numBodies; ++b) {
          const Body* body = e->bodies[b];
          const float dx = x - body->xf.p.x, dy = y - body->xf.p.y;
          const float d2 = dx * dx + dy * dy;
          const float R = (0.0165f + 0.002f) * S, Rin = (0.0165f + 0.002f - 0.005f) * S;
          if (d2 > R * R) continue;
          c[0] = c[1] = c[2] = 150.0f;
          if (d2 >= Rin * Rin) c[0] = c[1] = c[2] = 100.0f;
          if (sc.bodies[b].kind != KB_KILOBOT_SIMPLE_PHOTOTAXIS) {
            const float lx = body->xf.q.c * dx + body->xf.q.s * dy, ly = -body->xf.q.s * dx + body->xf.q.c * dy;
            const float front = (0.0165f - 0.005f) * S, hw = 0.0025f * S;
            if (lx >= 0.0f && lx <= front && ly >= -hw && ly <= hw) c[0] = c[1] = c[2] = 255.0f;
          }
        }
        for (int l = 0; l < h->numLights; ++l) {
          const KbLightDef& ld = sc.lights[l];
          if (ld.type == KB_LIGHT_LINEAR) continue;
          const LightState& ls = e->lights[l];
          const float lx = (float)(ls.pos[0] * 25.0), ly = (float)(ls.pos[1] * 25.0);
          const float R = (float)(ld.radius * 25.0);
          const float dx = x - lx, dy = y - ly;
          if (dx * dx + dy * dy <= R * R) {
            const float al = 150.0f / 255.0f, be = 1.0f - 150.0f / 255.0f;
            c[0] = 255.0f * al + c[0] * be;
            c[1] = 255.0f * al + c[1] * be;
            c[2] = 30.0f * al + c[2] * be;
          }
        }
        uint8_t* o = rgb + (((size_t)img * height + py) * width + px) * 3;
        for (int k = 0; k < 3; ++k) o[k] = (uint8_t)(int)(c[k] + 0.5f);
      }
  }
  return KB_OK;
}

int kbo_get_mass_data(KbHandle* hh, float* out) {
  Handle* h = reinterpret_cast<Handle*>(hh);
  // derived per scene by building a throw-away world at the origin
  const int B = h->numBodies;
  std::vector<double> pose((size_t)B * 3, 0.0);
  std::vector<double> light((size_t)std::max(1, h->lightStateDim), 0.0);
  for (size_t s = 0; s < h->scenes.size(); ++s) {
    Env tmp;
    tmp.scene = (int)s;
    // spread bodies far apart so that the settle step does nothing
    for (int b = 0; b < B; ++b) pose[3 * b] = 10.0 * (b + 1);
    Handle* hm = h;
    ResetEnv(hm, &tmp, pose.data(), light.data(), nullptr);
    for (int b = 0; b < B; ++b) {
      float* o = out + (s * B + b) * 4;
      o[0] = tmp.bodies[b]->invMass;
      o[1] = tmp.bodies[b]->invI;
      o[2] = tmp.bodies[b]->sweep.localCenter.x;
      o[3] = tmp.bodies[b]->sweep.localCenter.y;
    }
    delete tmp.world;
  }
  return KB_OK;
}

// direct access to the double-precision sincos used in place of libm sinf/cosf (tests only)
void kbo_sincosf(const float* a, float* s, float* c, int64_t n) {
  for (int64_t i = 0; i < n; ++i) SinCos(a[i], s + i, c + i);
}
void kbo_libm_sincosf(const float* a, float* s, float* c, int64_t n) {
  for (int64_t i = 0; i < n; ++i) {
    s[i] = sinf(a[i]);
    c[i] = cosf(a[i]);
  }
}


// ---- test hooks: evaluate single pieces of the Python-side restatement against golden vectors ----
// light.value_and_gradients at npts points for a (composite) light: state laid out like obs_light
void kbo_eval_light(const KbLightDef* defs, int32_t n, const double* state, const double* pts, int32_t npts,
                    double* value, double* grad) {
  for (int i = 0; i < npts; ++i) {
    double v = 0.0, gx = 0.0, gy = 0.0, best = 0.0;
    int off = 0;
    for (int l = 0; l < n; ++l) {
      LightState ls;
      if (defs[l].type == KB_LIGHT_LINEAR) ls.angle = state[off];
      else { ls.pos[0] = state[off]; ls.pos[1] = state[off + 1]; }
      double vv, g0, g1;
      LightValueGrad(defs[l], ls, pts[2 * i], pts[2 * i + 1], &vv, &g0, &g1);
      v += vv;
      if (l == 0 || vv > best) { best = vv; gx = g0; gy = g1; }
      off += LightStateDim(defs[l]);
    }
    value[i] = v;
    grad[2 * i] = gx;
    grad[2 * i + 1] = gy;
  }
}

// light.step: `substeps` calls with the same action; trace[substeps][dim]
void kbo_light_step(const KbLightDef* def, double* state, const double* action, int32_t substeps, double* trace) {
  LightState ls;
  const int dim = LightStateDim(*def);
  if (def->type == KB_LIGHT_LINEAR) ls.angle = state[0];
  else { ls.pos[0] = state[0]; ls.pos[1] = state[1]; if (dim == 4) { ls.vel[0] = state[2]; ls.vel[1] = state[3]; } }
  for (int s = 0; s < substeps; ++s) {
    LightStep(*def, &ls, action, 1. / 10);
    double* o = trace + (size_t)s * dim;
    if (def->type == KB_LIGHT_LINEAR) o[0] = ls.angle;
    else { o[0] = ls.pos[0]; o[1] = ls.pos[1]; if (dim == 4) { o[2] = ls.vel[0]; o[3] = ls.vel[1]; } }
  }
  if (def->type == KB_LIGHT_LINEAR) state[0] = ls.angle;
  else { state[0] = ls.pos[0]; state[1] = ls.pos[1]; if (dim == 4) { state[2] = ls.vel[0]; state[3] = ls.vel[1]; } }
}

// Kilobot.step on a free body at a fixed pose: `calls` controller calls, each fed (value, gx, gy);
// out[calls][3] = linearVelocity.x, linearVelocity.y, angularVelocity as handed to Box2D
void kbo_controller_trace(int32_t kind, float px, float py, float angle, const double* vel, const double* feed, int32_t calls,
                          float* out) {
  Handle h;
  ComputeMotorConstants(&h, 1. / 10);
  World w;
  w.CreateTable(-1000.f, -1000.f, 1000.f, 1000.f, 0, 0.2f);
  Body* b = w.CreateBody(px, py, angle, 0.8f, 0.8f);
  KilobotCtrl kc;
  kc.kind = kind;
  if (vel) { kc.velocity[0] = vel[0]; kc.velocity[1] = vel[1]; }
  for (int i = 0; i < calls; ++i) {
    kc.lightValue = feed[3 * i];
    kc.lightGrad[0] = feed[3 * i + 1];
    kc.lightGrad[1] = feed[3 * i + 2];
    RunController(&h, kc, b, 0.1f, 1. / 10);
    out[3 * i] = b->linearVelocity.x;
    out[3 * i + 1] = b->linearVelocity.y;
    out[3 * i + 2] = b->angularVelocity;
  }
}

// Kilobot.light_sensor_pos for a PhototaxisKilobot at the given pose (SI units in and out)
void kbo_sensor_pos(double x, double y, double angle, double* out) {
  Xf xf;
  xf.p.Set((float)(25.0 * x), (float)(25.0 * y));
  xf.q.Set((float)angle);
  Vec2 lp((float)(25.0 * 0.0), (float)(25.0 * -0.0165));
  Vec2 wp = Mul(xf, lp);
  out[0] = (double)wp.x / 25.0;
  out[1] = (double)wp.y / 25.0;
}

// Test-only probe of the narrowphase, distance and TOI routines (include/kb_b200.h kb_probe_geometry): the same layout,
// with the oracle's own shape code and the dispatch of Contact::Evaluate.
int kbo_probe_geometry(int32_t device, int32_t op, int32_t n, const KbProbeShape* shapes, int32_t num_shapes,
                       const KbProbeCase* cases, uint32_t* out) {
  (void)device;
  if (!shapes || num_shapes < 1 || !out || op < KB_PROBE_SHAPE || op > KB_PROBE_TOI || (op != KB_PROBE_SHAPE && (!cases || n < 0))) {
    g_err = "kbo_probe_geometry: invalid arguments";
    return KB_ERR_INVALID;
  }
  std::vector<Shape> sh((size_t)num_shapes);
  for (int s = 0; s < num_shapes; ++s) {
    const KbProbeShape& ps = shapes[s];
    if (ps.kind == KB_PROBE_EDGE) {
      if ((ps.wall_edges != 3 && ps.wall_edges != 4) || ps.edge < 0 || ps.edge >= ps.wall_edges) {
        g_err = "kbo_probe_geometry: bad chain edge";
        return KB_ERR_INVALID;
      }
      sh[s] = MakeChainEdge(ps.wall_x0, ps.wall_y0, ps.wall_x1, ps.wall_y1, ps.wall_edges, ps.edge);
    } else {
      sh[s] = MakeShape(ps.fixture);
    }
  }
  auto f2u = [](float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
  };
  if (op == KB_PROBE_SHAPE) {
    for (int s = 0; s < num_shapes; ++s) {
      const Shape& x = sh[s];
      uint32_t* o = out + (size_t)s * KB_PROBE_OUT_WORDS;
      std::memset(o, 0, KB_PROBE_OUT_WORDS * 4);
      o[0] = (uint32_t)(x.type == kEdge ? 2 : (x.type == kCircle ? 1 : x.count));
      o[1] = f2u(x.radius);
      o[2] = x.type == kEdge ? (uint32_t)x.hasVertex0 : 0u;
      o[3] = x.type == kEdge ? (uint32_t)x.hasVertex3 : 0u;
      if (x.type == kPolygon) {
        o[4] = f2u(x.centroid.x);
        o[5] = f2u(x.centroid.y);
        for (int i = 0; i < x.count; ++i) {
          o[6 + i] = f2u(x.vertices[i].x);
          o[14 + i] = f2u(x.vertices[i].y);
          o[22 + i] = f2u(x.normals[i].x);
          o[30 + i] = f2u(x.normals[i].y);
        }
      } else if (x.type == kEdge) {
        const Vec2 v[4] = {x.v0, x.v1, x.v2, x.v3};
        for (int i = 0; i < 4; ++i) {
          o[6 + i] = f2u(v[i].x);
          o[14 + i] = f2u(v[i].y);
        }
      }
    }
    return KB_OK;
  }
  for (int i = 0; i < n; ++i) {
    const KbProbeCase& c = cases[i];
    if (c.a < 0 || c.a >= num_shapes || c.b < 0 || c.b >= num_shapes) {
      g_err = "kbo_probe_geometry: shape index out of range";
      return KB_ERR_INVALID;
    }
    // the pairs the contact register forms (Contact::Evaluate): A a circle only against a circle, B never an edge
    const int tA = sh[c.a].type, tB = sh[c.b].type;
    if (op == KB_PROBE_COLLIDE && (tB == kEdge || (tA == kCircle && tB != kCircle))) {
      g_err = "kbo_probe_geometry: no narrowphase routine for this pair of shapes";
      return KB_ERR_INVALID;
    }
  }
  for (int i = 0; i < n; ++i) {
    const KbProbeCase& c = cases[i];
    const Shape* sA = &sh[c.a];
    const Shape* sB = &sh[c.b];
    uint32_t* o = out + (size_t)i * KB_PROBE_OUT_WORDS;
    std::memset(o, 0, KB_PROBE_OUT_WORDS * 4);
    Xf xfA, xfB;
    xfA.p.Set(c.xf_a[0], c.xf_a[1]);
    xfA.q.s = c.xf_a[2];
    xfA.q.c = c.xf_a[3];
    xfB.p.Set(c.xf_b[0], c.xf_b[1]);
    xfB.q.s = c.xf_b[2];
    xfB.q.c = c.xf_b[3];
    if (op == KB_PROBE_COLLIDE) {
      Manifold m;
      if (sA->type == kCircle && sB->type == kCircle) CollideCircles(&m, sA, xfA, sB, xfB);
      else if (sA->type == kPolygon && sB->type == kCircle) CollidePolygonAndCircle(&m, sA, xfA, sB, xfB);
      else if (sA->type == kPolygon && sB->type == kPolygon) CollidePolygons(&m, sA, xfA, sB, xfB);
      else if (sA->type == kEdge && sB->type == kCircle) CollideEdgeAndCircle(&m, sA, xfA, sB, xfB);
      else if (sA->type == kEdge && sB->type == kPolygon) CollideEdgeAndPolygon(&m, sA, xfA, sB, xfB);
      else m.pointCount = 0;
      o[0] = (uint32_t)m.type;
      o[1] = (uint32_t)m.pointCount;
      o[2] = f2u(m.localNormal.x);
      o[3] = f2u(m.localNormal.y);
      o[4] = f2u(m.localPoint.x);
      o[5] = f2u(m.localPoint.y);
      for (int k = 0; k < 2; ++k) {
        o[6 + 3 * k] = f2u(m.points[k].localPoint.x);
        o[7 + 3 * k] = f2u(m.points[k].localPoint.y);
        o[8 + 3 * k] = m.points[k].id.key;
      }
    } else if (op == KB_PROBE_DISTANCE) {
      int count = 0;
      o[0] = f2u(DistanceCore(sA, xfA, sB, xfB, &count));
      o[1] = (uint32_t)count;
    } else {
      TOIInput in;
      in.shapeA = sA;
      in.shapeB = sB;
      const float* w[2] = {c.sweep_a, c.sweep_b};
      Sweep* sw[2] = {&in.sweepA, &in.sweepB};
      for (int k = 0; k < 2; ++k) {
        sw[k]->localCenter.Set(w[k][0], w[k][1]);
        sw[k]->c0.Set(w[k][2], w[k][3]);
        sw[k]->c.Set(w[k][4], w[k][5]);
        sw[k]->a0 = w[k][6];
        sw[k]->a = w[k][7];
        sw[k]->alpha0 = 0.0f;
      }
      in.tMax = 1.0f;
      TOIOutput res;
      TimeOfImpact(&res, &in);
      const float t = res.state == TOIOutput::kTouching ? res.t : -1.0f;
      o[0] = f2u(t);
      o[1] = (sA->type == kEdge && sB->type == kCircle) ? f2u(t) : 0u;
      o[2] = f2u(t);
      o[3] = (uint32_t)res.state;
    }
  }
  return KB_OK;
}

}  // extern "C"
