// CPU ORACLE WITH THE ACTUATION MODEL -- TEST INFRASTRUCTURE ONLY (built by tests/test_actuation.py into a temporary
// directory).
//
// The oracle under oracle/ restates the reference and is not changed by the actuation model (include/kb_b200.h
// kb_set_actuation), an extension beyond it.  This file builds that same oracle -- oracle/kbo_env.cpp is included
// below, unchanged -- with the model on top, as an independent restatement of what the kernels do:
//   - every velocity a kilobot controller hands to Box2D (RunController's b->SetLinearVelocity / SetAngularVelocity,
//     whose body is named `b` there) goes through kbo_act::Linear / Angular, which scale it by the kilobot's draws and
//     sub-step noise, add the drift, or -- for a dead kilobot -- drop the call, so that the body stays passive;
//   - kbo_create's handles get kbo_set_actuation / kbo_get_actuation, kbo_reset advances the reset envs' actuation
//     episode and redraws them, kbo_step counts the env-steps the noise is keyed by.
// A body the model does not know (no model attached, kbo_controller_trace's free body) takes the plain call, so this
// library computes exactly what oracle/libkbo.so computes until kbo_set_actuation is called.
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../oracle/kbo_world.h"

namespace kbo_act {
void Linear(kbo::Body* b, const kbo::Vec2& v);
void Angular(kbo::Body* b, float w);
}  // namespace kbo_act

// the wrapped entry points keep their names; the originals are compiled under these
#define kbo_destroy kbo_destroy_base
#define kbo_reset kbo_reset_base
#define kbo_step kbo_step_base
#define kbo_step_host kbo_step_host_base
// the controllers' velocity commands (the left operand only keeps `b->` well-formed)
#define SetLinearVelocity(v) linearVelocity, ::kbo_act::Linear(b, v)
#define SetAngularVelocity(w) angularVelocity, ::kbo_act::Angular(b, w)
#include "../oracle/kbo_env.cpp"
#undef SetLinearVelocity
#undef SetAngularVelocity
#undef kbo_destroy
#undef kbo_reset
#undef kbo_step
#undef kbo_step_host

namespace kbo_act {

// Philox4x32-10 as gym_kilobots_b200/philox.py and csrc/kb_sample.cuh evaluate it
struct Philox4 {
  uint32_t x, y, z, w;
};
static Philox4 Philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}
static double U53(uint32_t hi, uint32_t lo) {
  return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) / 9007199254740992.0;
}
static const uint32_t kStreamActuation = 9, kStreamActuationNoise = 10;

// the actuation model of one handle
struct State {
  kbo::Handle* h = nullptr;
  KbActuationDef def = {};
  uint64_t step = 0;                     // kbo_step calls since kbo_set_actuation
  std::vector<uint32_t> episode;         // [E]
  std::vector<std::vector<float>> draws;   // [E][N * 4] = (g_v, g_w, d_w, alive)
  std::vector<uint64_t> substepBase;     // [E] the env's world sub-step count when the current env-step began
  std::vector<std::vector<kbo::Body*>> bodies;   // [E] the kilobot bodies registered for the env
};
struct Slot {
  State* st;
  int env, k;
};
static std::mutex g_mu;   // guards the two maps; steps only read them
static std::unordered_map<const kbo::Handle*, State*> g_states;
static std::unordered_map<const kbo::Body*, Slot> g_bodies;

static void Draw(State* st, int i) {
  const KbActuationDef& d = st->def;
  const uint64_t g = (uint64_t)(d.env_id_base + i);
  const int N = st->h->numKilobots;
  const uint32_t k0 = (uint32_t)d.seed, k1 = (uint32_t)(d.seed >> 32), c1 = kStreamActuation + (st->episode[i] << 8);
  std::vector<float>& out = st->draws[i];
  out.assign((size_t)N * 4, 0.0f);
  for (int k = 0; k < N; ++k) {
    const Philox4 a = Philox4x32(2u * (uint32_t)k, c1, (uint32_t)g, (uint32_t)(g >> 32), k0, k1);
    const Philox4 b = Philox4x32(2u * (uint32_t)k + 1u, c1, (uint32_t)g, (uint32_t)(g >> 32), k0, k1);
    float* o = out.data() + 4 * k;
    o[0] = (float)(d.gain_v_lo + (d.gain_v_hi - d.gain_v_lo) * U53(a.x, a.y));
    o[1] = (float)(d.gain_w_lo + (d.gain_w_hi - d.gain_w_lo) * U53(a.z, a.w));
    o[2] = (float)(d.drift_w * (2.0 * U53(b.x, b.y) - 1.0));
    o[3] = U53(b.z, b.w) < d.p_dead ? 0.0f : 1.0f;
  }
}

// (re)register the kilobot bodies of env i (its world is rebuilt by every reset); caller holds g_mu
static void Bind(State* st, int i) {
  for (kbo::Body* b : st->bodies[i]) g_bodies.erase(b);
  st->bodies[i].clear();
  const kbo::Env& e = st->h->envs[i];
  if (!e.world) return;
  for (int k = 0; k < st->h->numKilobots; ++k) {
    kbo::Body* b = e.bodies[st->h->numObjects + k];
    st->bodies[i].push_back(b);
    g_bodies[b] = Slot{st, i, k};
  }
}

static void Unbind(State* st) {
  for (auto& v : st->bodies)
    for (kbo::Body* b : v) g_bodies.erase(b);
}

struct Factors {
  float gv, gw, dw, fv, fw;
  bool alive, drift;
};
// the draws and this sub-step's noise factors of the kilobot of body b; false: no model acts on b
static bool Lookup(const kbo::Body* b, Factors* f) {
  const auto it = g_bodies.find(b);
  if (it == g_bodies.end()) return false;
  const Slot& s = it->second;
  const State* st = s.st;
  const KbActuationDef& d = st->def;
  const float* dr = st->draws[s.env].data() + 4 * s.k;
  f->gv = dr[0];
  f->gw = dr[1];
  f->dw = dr[2];
  f->alive = dr[3] != 0.0f;
  f->drift = d.drift_w > 0.0;
  f->fv = f->fw = 1.0f;
  if (d.noise_v > 0.0 || d.noise_w > 0.0) {
    const uint32_t sub = (uint32_t)(st->h->envs[s.env].world->counters.substeps - st->substepBase[s.env]);
    const uint64_t g = (uint64_t)(d.env_id_base + s.env);
    const Philox4 r = Philox4x32((uint32_t)s.k | (sub << 16), (uint32_t)st->step, (uint32_t)g,
                                 kStreamActuationNoise | ((uint32_t)(g >> 32) << 8), (uint32_t)d.seed,
                                 (uint32_t)(d.seed >> 32));
    f->fv = (float)(1.0 + d.noise_v * (2.0 * U53(r.x, r.y) - 1.0));
    f->fw = (float)(1.0 + d.noise_w * (2.0 * U53(r.z, r.w) - 1.0));
  }
  return true;
}

void Linear(kbo::Body* b, const kbo::Vec2& v) {
  Factors f;
  if (!Lookup(b, &f)) {
    b->SetLinearVelocity(v);
  } else if (f.alive) {
    b->SetLinearVelocity(kbo::Vec2((v.x * f.gv) * f.fv, (v.y * f.gv) * f.fv));
  }
}

void Angular(kbo::Body* b, float w) {
  Factors f;
  if (!Lookup(b, &f)) {
    b->SetAngularVelocity(w);
  } else if (f.alive) {
    w = (w * f.gw) * f.fw;
    b->SetAngularVelocity(f.drift ? w + f.dw : w);
  }
}

static State* Find(const kbo::Handle* h) {
  const auto it = g_states.find(h);
  return it == g_states.end() ? nullptr : it->second;
}

}  // namespace kbo_act

extern "C" {

int kbo_destroy(KbHandle* hh) {
  {
    std::lock_guard<std::mutex> lock(kbo_act::g_mu);
    if (kbo_act::State* st = kbo_act::Find(reinterpret_cast<kbo::Handle*>(hh))) {
      kbo_act::Unbind(st);
      kbo_act::g_states.erase(st->h);
      delete st;
    }
  }
  return kbo_destroy_base(hh);
}

int kbo_reset(KbHandle* hh, const uint8_t* mask, const double* body_pose, const double* light_state,
              const double* kb_velocity, void* stream) {
  const int rc = kbo_reset_base(hh, mask, body_pose, light_state, kb_velocity, stream);
  std::lock_guard<std::mutex> lock(kbo_act::g_mu);
  kbo_act::State* st = kbo_act::Find(reinterpret_cast<kbo::Handle*>(hh));
  if (!st) return rc;
  for (int i = 0; i < (int)st->episode.size(); ++i) {
    if (mask && !mask[i]) continue;
    st->episode[i] += 1u;   // the env's next actuation episode
    kbo_act::Draw(st, i);
    kbo_act::Bind(st, i);
  }
  return rc;
}

int kbo_step(KbHandle* hh, const double* action, int32_t action_mode, float* obs_kilobots, float* obs_objects,
             double* obs_light, float* reward, uint8_t* done, int32_t* status, void* stream) {
  kbo_act::State* st;
  {
    std::lock_guard<std::mutex> lock(kbo_act::g_mu);
    st = kbo_act::Find(reinterpret_cast<kbo::Handle*>(hh));
  }
  if (st)
    for (size_t i = 0; i < st->substepBase.size(); ++i)
      st->substepBase[i] = st->h->envs[i].world ? st->h->envs[i].world->counters.substeps : 0;
  const int rc = kbo_step_base(hh, action, action_mode, obs_kilobots, obs_objects, obs_light, reward, done, status, stream);
  if (st) ++st->step;
  return rc;
}

int kbo_step_host(KbHandle* hh, const double* action, int32_t action_mode, float* obs_kilobots, float* obs_objects,
                  double* obs_light, float* reward, uint8_t* done, int32_t* status, void* stream) {
  return kbo_step(hh, action, action_mode, obs_kilobots, obs_objects, obs_light, reward, done, status, stream);
}

// include/kb_b200.h kb_set_actuation: same semantics and refusals
int kbo_set_actuation(KbHandle* hh, const KbActuationDef* def) {
  kbo::Handle* h = reinterpret_cast<kbo::Handle*>(hh);
  std::lock_guard<std::mutex> lock(kbo_act::g_mu);
  kbo_act::State* st = kbo_act::Find(h);
  if (!def) {
    if (st) {
      kbo_act::Unbind(st);
      kbo_act::g_states.erase(h);
      delete st;
    }
    return KB_OK;
  }
  const KbActuationDef& d = *def;
  const struct {
    const char* name;
    double v;
  } fields[] = {{"gain_v_lo", d.gain_v_lo}, {"gain_v_hi", d.gain_v_hi}, {"gain_w_lo", d.gain_w_lo}, {"gain_w_hi", d.gain_w_hi},
                {"drift_w", d.drift_w},     {"noise_v", d.noise_v},     {"noise_w", d.noise_w},     {"p_dead", d.p_dead}};
  for (const auto& f : fields) {
    if (!std::isfinite(f.v)) return kbo::g_err = std::string("kbo_set_actuation: ") + f.name + " is not finite", KB_ERR_INVALID;
    if (f.v < 0.0) return kbo::g_err = std::string("kbo_set_actuation: ") + f.name + " is negative", KB_ERR_INVALID;
  }
  if (d.gain_v_lo > d.gain_v_hi) return kbo::g_err = "kbo_set_actuation: gain_v_lo > gain_v_hi", KB_ERR_INVALID;
  if (d.gain_w_lo > d.gain_w_hi) return kbo::g_err = "kbo_set_actuation: gain_w_lo > gain_w_hi", KB_ERR_INVALID;
  if (d.p_dead > 1.0) return kbo::g_err = "kbo_set_actuation: p_dead is outside [0, 1]", KB_ERR_INVALID;
  if (st) kbo_act::Unbind(st);
  else st = kbo_act::g_states[h] = new kbo_act::State();
  const size_t E = h->envs.size();
  st->h = h;
  st->def = d;
  st->step = 0;
  st->episode.assign(E, 0u);
  st->draws.assign(E, std::vector<float>());
  st->substepBase.assign(E, 0);
  st->bodies.assign(E, std::vector<kbo::Body*>());
  for (int i = 0; i < (int)E; ++i) {   // episode 0 of every env
    kbo_act::Draw(st, i);
    kbo_act::Bind(st, i);
  }
  return KB_OK;
}

int kbo_get_actuation(KbHandle* hh, float* draws, uint32_t* episodes, uint64_t* step) {
  std::lock_guard<std::mutex> lock(kbo_act::g_mu);
  const kbo_act::State* st = kbo_act::Find(reinterpret_cast<kbo::Handle*>(hh));
  if (!st) {
    kbo::g_err = "kbo_get_actuation: no actuation model (kbo_set_actuation)";
    return KB_ERR_INVALID;
  }
  const size_t N = (size_t)st->h->numKilobots;
  for (size_t i = 0; i < st->episode.size(); ++i) {
    if (draws) std::memcpy(draws + i * N * 4, st->draws[i].data(), sizeof(float) * N * 4);
    if (episodes) episodes[i] = st->episode[i];
  }
  if (step) *step = st->step;
  return KB_OK;
}

}  // extern "C"
