// kb_env.cuh -- the environment layer around the physics, written once for both kernel tiers: lights
// (lib/light.py:59-75,176-189,237-253,300-316), kilobot controllers (lib/kilobot.py:54-55,86-127,188-203,253-258,
// 294-300,307-316,318-333) and the task layer (include/kb_b200.h "Task layer").
//
// Every function is a template over the tier's simulation struct T -- Sim<LPE, UNI, LT> (kb_step.cuh, a lane group per
// env) or Swarm<NT> (kb_swarm.cuh, a CTA per env) -- and reaches it through the members both define: L, bc,
// lightState(), lightConst(l), ctrl(k), bodyXf(b), pos4(b), vel4(b), wake(b), bkind(b), hdr(i) and obsPos(b), the
// position the task and the observations read.  Kilobot k is body L.M + k.  The caller picks the thread (single-thread
// functions) or passes its (first, stride) pair (per-kilobot loops), and issues every barrier itself.
//
// Included by kb_step.cuh once KernelArgs is declared.
#pragma once

namespace kb {

__device__ __forceinline__ double clipd(double a, double lo, double hi) {
  double m = a > lo ? a : lo;
  return m < hi ? m : hi;
}

// one light step of every light from the env's light action (single thread)
template <class T>
__device__ __forceinline__ void lightStep(T& s, const double* action) {
  const SF64Arr ls = s.lightState();
  int so = 0, ao = 0;
  for (int l = 0; l < s.L.numLights; ++l) {
    const LCs lc = s.lightConst(l);
    const int lt = lc.type();
    if (lt == KB_LIGHT_CIRCULAR) {
      double a0 = clipd(action[ao], lc.alo(0), lc.ahi(0));
      double a1 = clipd(action[ao + 1], lc.alo(1), lc.ahi(1));
      const double dt = 1. / 10;
      if (lc.relative()) {
        ls[so] += a0 * dt;
        ls[so + 1] += a1 * dt;
      } else {
        ls[so] = a0;
        ls[so + 1] = a1;
      }
      ls[so] = clipd(ls[so], lc.blo(0), lc.bhi(0));
      ls[so + 1] = clipd(ls[so + 1], lc.blo(1), lc.bhi(1));
      so += 2;
      ao += 2;
    } else if (lt == KB_LIGHT_MOMENTUM) {
      const double dt = 1. / 10;
      double a0 = clipd(action[ao], lc.alo(0), lc.ahi(0));
      double a1 = clipd(action[ao + 1], lc.alo(1), lc.ahi(1));
      ls[so + 2] += a0 * dt;
      ls[so + 3] += a1 * dt;
      const double v2 = ls[so + 2], v3 = ls[so + 3];
      double n = sqrt(v2 * v2 + v3 * v3);
      const double mv = lc.maxVel();
      if (n > mv) {
        double f = mv / n;
        ls[so + 2] *= f;
        ls[so + 3] *= f;
      }
      ls[so] += (double)ls[so + 2] * dt;
      ls[so + 1] += (double)ls[so + 3] * dt;
      ls[so] = clipd(ls[so], lc.blo(0), lc.bhi(0));
      ls[so + 1] = clipd(ls[so + 1], lc.blo(1), lc.bhi(1));
      so += 4;
      ao += 2;
    } else {
      double a = clipd(action[ao], lc.alo(0), lc.ahi(0));
      const double pi = 3.141592653589793;
      if (a < -pi) a += 2 * pi;
      if (a > pi) a -= 2 * pi;
      ls[so] = a;
      so += 1;
      ao += 1;
    }
  }
}

__device__ __forceinline__ void lightValueGrad(const LCs lc, const SF64Arr ls, double sx, double sy, double* value,
                                               double* gx, double* gy) {
  if (lc.type() == KB_LIGHT_LINEAR) {
    const double2 sc = kb_sincosd(ls[0]);
    const double vx = sc.y, vy = sc.x;
    *value = vx * sx + vy * sy;
    *gx = vx;
    *gy = vy;
    return;
  }
  double g0 = -1 * (sx - (double)ls[0]);
  double g1 = -1 * (sy - (double)ls[1]);
  double norm = sqrt(g0 * g0 + g1 * g1);
  double v = 1.0;
  const double radius = lc.radius();
  v -= norm / radius;
  v = v < 1. ? v : 1.;
  v = v > .0 ? v : .0;
  v *= 255;
  if (norm == 0.0) {
    g0 = 0.0;
    g1 = 0.0;
  } else {
    g0 /= norm;
    g1 /= norm;
  }
  if (norm > radius) {
    g0 *= .0;
    g1 *= .0;
  }
  *value = v;
  *gx = g0;
  *gy = g1;
}

// b2Body::SetLinearVelocity / SetAngularVelocity on a kilobot from the thread that owns it
template <class T>
__device__ __forceinline__ void setLinearVelocity(T& s, int b, V2 v) {
  if (dot(v, v) > 0.0f) s.wake(b);
  s.vel4(b).set(0, v.x);
  s.vel4(b).set(1, v.y);
}
template <class T>
__device__ __forceinline__ void setAngularVelocity(T& s, int b, float w) {
  if (w * w > 0.0f) s.wake(b);
  s.vel4(b).set(2, w);
}

// Kilobot.set_action of every velocity / acceleration kilobot (action == null: zero action).  An absent kilobot's kind
// (KB_BODY_ABSENT) takes neither branch: its action row is never read and may hold anything.
template <class T>
__device__ __forceinline__ void setKilobotActions(T& s, const double* action, int first, int stride) {
  const double hpi = 0.5 * 3.141592653589793;
  const double pi = 3.141592653589793;
#pragma unroll 1
  for (int k = first; k < s.L.N; k += stride) {
    const int kind = s.bkind(s.L.M + k);
    double* c = s.ctrl(k);
    const double* a = action ? action + 2 * k : nullptr;
    if (kind == KB_KILOBOT_VELOCITY) {
      if (a) {
        c[0] = clipd(a[0], .0, 0.01);
        c[1] = clipd(a[1], -hpi, hpi);
      } else {
        c[0] = .0;
        c[1] = .0;
      }
    } else if (kind == KB_KILOBOT_ACCELERATION) {
      if (a) {
        c[2] = clipd(a[0], -.005, .005);
        c[3] = clipd(a[1], -.2 * pi, .2 * pi);
      } else {
        c[2] = .0;
        c[3] = .0;
      }
    }
  }
}

// every kilobot senses the light and runs its controller, which sets its velocity (an absent kilobot neither senses nor
// runs a controller: KB_BODY_ABSENT needs no light and takes the default case)
template <class T>
__device__ __forceinline__ void senseControl(T& s, int first, int stride) {
  const auto& L = s.L;
  const SF64Arr ls = s.lightState();
#pragma unroll 1
  for (int k = first; k < L.N; k += stride) {
    const int b = L.M + k;
    const int kind = s.bkind(b);
    const Xf xf = s.bodyXf(b);
    double* c = s.ctrl(k);
    double value = 0.0, gx = 0.0, gy = 0.0;
    // the light is only looked at where its value can reach the controller: a PhototaxisKilobot samples
    // on every 6th call (lib/kilobot.py:328-333), velocity / acceleration control never
    const bool needLight = kind == KB_KILOBOT_SIMPLE_PHOTOTAXIS || (kind == KB_KILOBOT_PHOTOTAXIS && ((int)c[2] % 6) == 0);
    if (L.numLights > 0 && needLight) {
      double sx, sy;
      if (kind == KB_KILOBOT_SIMPLE_PHOTOTAXIS) {
        sx = (double)xf.p.x / 25.0;
        sy = (double)xf.p.y / 25.0;
      } else {
        V2 lp = mk((float)(25.0 * 0.0), (float)(25.0 * -0.0165));
        V2 wp = xmul(xf, lp);
        sx = (double)wp.x / 25.0;
        sy = (double)wp.y / 25.0;
      }
      if (L.numLights == 1) {
        lightValueGrad(s.lightConst(0), ls, sx, sy, &value, &gx, &gy);
      } else {
        double best = 0.0;
        int so = 0;
        for (int l = 0; l < L.numLights; ++l) {
          double v, g0, g1;
          lightValueGrad(s.lightConst(l), ls + so, sx, sy, &v, &g0, &g1);
          value += v;
          if (l == 0 || v > best) {
            best = v;
            gx = g0;
            gy = g1;
          }
          const int lt = s.lightConst(l).type();
          so += lt == KB_LIGHT_MOMENTUM ? 4 : (lt == KB_LIGHT_LINEAR ? 1 : 2);
        }
      }
    }
    switch (kind) {
      case KB_KILOBOT_PHOTOTAXIS: {
        // c[0] threshold, c[1] turnRight, c[2] updateCounter, c[3] noChangeCounter
        int upd = (int)c[2];
        int turnRight = (int)c[1];
        if (upd % 6) {
          upd += 1;
        } else {
          upd += 1;
          int noChange = (int)c[3];
          if (value > c[0] || noChange >= 15) {
            c[0] = value + .01;
            turnRight = turnRight ? 0 : 1;
            noChange = 0;
          } else {
            noChange += 1;
          }
          c[3] = (double)noChange;
          c[1] = (double)turnRight;
        }
        c[2] = (double)upd;
        const float tx = turnRight ? L.transRight[0] : L.transLeft[0];
        const float ty = turnRight ? L.transRight[1] : L.transLeft[1];
        const float w = turnRight ? L.omegaRight : L.omegaLeft;
        V2 wv = rmul(xf.q, mk(tx, ty));
        V2 lv = mk(wv.x / 25.0f, wv.y / 25.0f);
        lv = mk(lv.x / L.dt, lv.y / L.dt);
        lv = mk(lv.x * 25.0f, lv.y * 25.0f);
        setAngularVelocity(s, b, w);
        setLinearVelocity(s, b, lv);
      } break;
      case KB_KILOBOT_SIMPLE_PHOTOTAXIS: {
        double mx = gx, my = gy;
        double n = sqrt(mx * mx + my * my);
        if (n > 0.01) {
          mx = mx / n * 0.01;
          my = my / n * 0.01;
        }
        mx *= 25.0;
        my *= 25.0;
        setLinearVelocity(s, b, mk((float)mx, (float)my));
        // linearDamping = 0: kept as a per-kind constant of the solver's damping
      } break;
      case KB_KILOBOT_ACCELERATION: {
        const double hpi = 0.5 * 3.141592653589793;
        const double dt = 1. / 10;
        c[0] += c[2] * dt;
        c[1] += c[3] * dt;
        c[0] = c[0] > .0 ? c[0] : .0;
        c[1] = c[1] > -hpi ? c[1] : -hpi;
        c[0] = c[0] < 0.01 ? c[0] : 0.01;
        c[1] = c[1] < hpi ? c[1] : hpi;
      }  // fallthrough
      case KB_KILOBOT_VELOCITY: {
        double ang = (double)s.pos4(b).get(2);
        const double2 sc = kb_sincosd(ang);
        double lx = sc.y, ly = sc.x;
        lx *= c[0] * 25.0;
        ly *= c[0] * 25.0;
        setLinearVelocity(s, b, mk((float)lx, (float)ly));
        setAngularVelocity(s, b, (float)c[1]);
      } break;
      default: break;
    }
  }
}

// ------------------------------------------------------------------------------------------------- task layer
// The scene the env was last reset with (kb_set_env_scene takes effect at the next reset).
template <class T>
__device__ __forceinline__ int envSceneOf(T& s, const KernelArgs& a) {
  return a.envScene ? (int)s.hdr(H_SCENE) : 0;
}

// distance (m) and |angle| (rad) between the task's subject and its target, float64, sequential sums -- the oracle
// evaluates the same expressions in the same order (oracle/kbo_env.cpp TaskError).  n: the kilobots of the env's
// scene (bodies L.M .. L.M + n - 1; in a batch of one size n == L.N).
template <class T>
__device__ __forceinline__ void taskError(T& s, const TaskConst& tk, const double* tgt, int n, double* dist, double* ang) {
  const auto& L = s.L;
  double px, py, th = 0.0;
  if (tk.mode == KB_TASK_OBJECT_TO_TARGET) {
    const float2 x = s.obsPos(tk.object);
    px = (double)x.x / 25.0;
    py = (double)x.y / 25.0;
    th = (double)s.pos4(tk.object).get(2);
  } else {
    double sx = 0.0, sy = 0.0;
    for (int b = L.M; b < L.M + n; ++b) {
      const float2 x = s.obsPos(b);
      sx += (double)x.x / 25.0;
      sy += (double)x.y / 25.0;
    }
    px = sx / (double)n;
    py = sy / (double)n;
  }
  const double dx = px - tgt[0], dy = py - tgt[1];
  *dist = sqrt(dx * dx + dy * dy);
  *ang = tk.mode == KB_TASK_OBJECT_TO_TARGET ? fabs(remainder(th - tgt[2], 6.283185307179586)) : 0.0;
}

// task error before the env-step, kept in the env's task words (not in registers) until taskEnd (single thread)
template <class T>
__device__ __forceinline__ void taskBegin(T& s, const KernelArgs& a, int env) {
  double* ts = a.taskState + (size_t)env * KB_TASK_WORDS;
  const int n = __ldg(&a.scenes[envSceneOf(s, a)].numKilobots);
  double d0, a0;
  taskError(s, a.task, ts, n, &d0, &a0);
  ts[3 + KB_EPISODE_STATS] = d0;
  ts[3 + KB_EPISODE_STATS + 1] = a0;
}

// get_state's light part (kilobots_env.py:115-118): the light state into the light and the flat observation
template <class T>
__device__ __forceinline__ void observeLights(T& s, const KernelArgs& a, int env, float* flat, int first, int stride) {
  const auto& L = s.L;
  if (a.obsLight || flat) {
    const SF64Arr ls = s.lightState();
#pragma unroll 1
    for (int i = first; i < L.L; i += stride) {
      const double v = ls[i];
      if (a.obsLight) a.obsLight[(size_t)env * L.L + i] = v;
      if (flat) flat[2 * L.N + i] = (float)v;
    }
  }
}

// the reward / done / info hooks (kilobots_env.py:123-131): reward, done, episode statistics, status (single thread)
template <class T>
__device__ __forceinline__ void taskEnd(T& s, const KernelArgs& a, int env) {
  const SceneConst* sc = a.scenes + envSceneOf(s, a);
  float rew = __ldg(&sc->rewardConst);
  uint8_t dn = 0;
  if (a.task.mode != KB_TASK_CONST) {
    double* ts = a.taskState + (size_t)env * KB_TASK_WORDS;
    double d1, a1;
    taskError(s, a.task, ts, __ldg(&sc->numKilobots), &d1, &a1);
    const double d0 = ts[3 + KB_EPISODE_STATS], a0 = ts[3 + KB_EPISODE_STATS + 1];  // stashed by taskBegin
    const bool success = d1 <= a.task.posTol && a1 <= a.task.angTol;
    double r = a.task.wPos * (d0 - d1);
    r = r + a.task.wAng * (a0 - a1);
    r = r - a.task.stepPenalty;
    if (success) r = r + a.task.bonus;
    const double len = ts[3 + KB_EP_LENGTH] + 1.0;
    dn = (success || (a.task.maxSteps > 0 && len >= (double)a.task.maxSteps)) ? 1 : 0;
    ts[3 + KB_EP_RETURN] += r;
    ts[3 + KB_EP_LENGTH] = len;
    ts[3 + KB_EP_POSITION_ERROR] = d1;
    ts[3 + KB_EP_ORIENTATION_ERROR] = a1;
    ts[3 + KB_EP_SUCCESS] = success ? 1.0 : 0.0;
    if (dn) ts[3 + KB_EP_DONE_COUNT] += 1.0;
    rew = (float)r;
  }
  if (a.reward) a.reward[env] = rew;
  if (a.done) a.done[env] = dn;
  if (a.status) a.status[env] = (int32_t)s.hdr(H_STATUS);
}

// reset of the environment layer: a new episode's task words, light.__init__ / MomentumLight(velocity=...) /
// GradientLight(angle=...), and the controllers (PhototaxisKilobot.__init__ lib/kilobot.py:307-316: threshold -inf,
// turn_left; velocity / acceleration kilobots start at kbVel).  env: the env's slot, envIn: the row of its inputs.
// The kinds are read from the scene's body constants: a tier's own copy of them may not be written yet.
template <class T>
__device__ __forceinline__ void resetEnvLayer(T& s, const KernelArgs& a, int env, int envIn, int first, int stride) {
  const auto& L = s.L;
  if (first == 0 && a.taskState && env < a.numEnvs) {
    double* ts = a.taskState + (size_t)env * KB_TASK_WORDS;
    ts[3 + KB_EP_RETURN] = 0.0;
    ts[3 + KB_EP_LENGTH] = 0.0;
    ts[3 + KB_EP_SUCCESS] = 0.0;
  }
  for (int i = first; i < L.L; i += stride) s.lightState()[i] = a.lightInit ? a.lightInit[(size_t)envIn * L.L + i] : 0.0;
  for (int k = first; k < L.N; k += stride) {
    double* c = s.ctrl(k);
    const int kind = __ldg(&s.bc[L.M + k].kind);
    c[0] = c[1] = c[2] = c[3] = 0.0;
    if (kind == KB_KILOBOT_PHOTOTAXIS) {
      c[0] = __longlong_as_double(0xFFF0000000000000LL);  // -inf
    } else if ((kind == KB_KILOBOT_VELOCITY || kind == KB_KILOBOT_ACCELERATION) && a.kbVel) {
      c[0] = a.kbVel[((size_t)envIn * L.N + k) * 2 + 0];
      c[1] = a.kbVel[((size_t)envIn * L.N + k) * 2 + 1];
    }
  }
}

}  // namespace kb
