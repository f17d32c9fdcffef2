// tests/emul/emul.cpp - TEST INFRASTRUCTURE: compiles the device code (csrc/dg_env.cuh, dg_ray.cuh, dg_dyn.cuh, dg_ik.cuh) with g++
// so that the kernel logic can be checked against the fp64 oracle and references in the GPU-less container.  A team of `nt` lanes
// is emulated by running every phase lane after lane (the barrier semantics of the GPU schedule); the ray, dynamics and IK kernels
// are emulated one environment after another.  Never shipped, never used by the product path: diy_gym_b200 raises when
// libdiygym_b200.so / a CUDA device is missing.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../diy_gym_b200/csrc/dg_env.cuh"
#include "../../diy_gym_b200/csrc/dg_ray.cuh"
#include "../../diy_gym_b200/csrc/dg_dyn.cuh"
#include "../../diy_gym_b200/csrc/dg_ik.cuh"

using namespace dg;

struct EmulWorld {
  HostScene hs;
  int n_envs, team;
  std::vector<float> state, param, ws, wg;
  uint32_t seed = 1234u; int env_off = 0;
  unsigned long long opmask[2] = {~0ull, ~0ull};
  unsigned dropped = 0;
};

template <int MAXD, int M>
static void ik_solve_all(const DevScene& d, const IkArgs& a, const float* state, int n_envs) {
  std::vector<float> scr(IkFastScratch<MAXD>::floats);
  for (int e = 0; e < n_envs; e++) ik_env<MAXD, M>(row_env(d, a.rec + (size_t)e * a.rec_stride), a, state + (size_t)e * d.S, e, scr.data());
}

extern "C" {
EmulWorld* dge_create(const int32_t* ibuf, int ni, const double* fbuf, int nf, int n_envs, int team, int ws_mode) {
  EmulWorld* w = new EmulWorld();
  if (!w->hs.build(ibuf, ni, fbuf, nf, team, ws_mode)) { fprintf(stderr, "emul: %s\n", w->hs.error.c_str()); delete w; return nullptr; }
  w->n_envs = n_envs; w->team = team;
  if (const char* es = getenv("DG_SOLVER")) w->hs.dev.solver = atoi(es) != 0;
  if (const char* em = getenv("DG_RS_MIN")) w->hs.dev.rs_min = atoi(em);
  const DevScene& d = w->hs.dev;
  w->state.resize((size_t)n_envs * d.S + 1); w->param.resize((size_t)n_envs * d.P + 1); w->ws.assign((size_t)d.w_total + 16, 0.f); w->wg.assign((size_t)d.g_total + 16, 0.f);
  for (int e = 0; e < n_envs; e++) {
    for (int i = 0; i < d.S; i++) w->state[(size_t)e * d.S + i] = d.state_def[i];
    for (int i = 0; i < d.P; i++) w->param[(size_t)e * d.P + i] = d.param_def[i];
  }
  return w;
}
void dge_destroy(EmulWorld* w) { delete w; }
float* dge_state(EmulWorld* w) { return w->state.data(); }
float* dge_param(EmulWorld* w) { return w->param.data(); }
int dge_ws_floats(EmulWorld* w) { return w->hs.dev.w_total; }
int dge_cold_floats(EmulWorld* w) { return w->hs.dev.g_total; }
void dge_set_action_mask(EmulWorld* w, const uint8_t* en, int n) { w->opmask[0] = w->opmask[1] = ~0ull; for (int k = 0; k < n && k < 128; k++) if (!en[k]) w->opmask[k >> 6] &= ~(1ull << (k & 63)); }
void dge_set_seed(EmulWorld* w, uint32_t seed, int env_off) { w->seed = seed; w->env_off = env_off; }
static Env make_env(EmulWorld* w, int e, const float* act, float* obs, float* rew, uint8_t* term) {
  const DevScene& d = w->hs.dev;
  Env C = row_env(d, w->state.data() + (size_t)e * d.S);
  C.ws = w->ws.data(); C.wg = w->wg.data(); C.pr = w->param.data() + (size_t)e * d.P;
  C.act = act ? act + (size_t)e * d.n_act : nullptr; C.obs = obs + (size_t)e * d.n_obs; C.rew = rew + (size_t)e * d.n_rew; C.term = term + (size_t)e * d.n_term;
  C.active = true; C.grp1 = 1; C.dropped = &w->dropped; C.e_local = e; C.seed = w->seed; C.env_id = w->env_off + e; C.opmask[0] = w->opmask[0]; C.opmask[1] = w->opmask[1];
  return C;
}
// DGE_POISON=<value>: fills both workspaces with that value before every environment, so that a read of workspace memory
// that this step did not write (garbage on the GPU, zeros here otherwise) shows up as a changed result
static void poison(EmulWorld* w) { if (const char* p = getenv("DGE_POISON")) { float v = (float)atof(p); for (auto& x : w->ws) x = v; for (auto& x : w->wg) x = v; } }
void dge_step(EmulWorld* w, const float* act, float* obs, float* rew, uint8_t* term) {
  for (int e = 0; e < w->n_envs; e++) { poison(w); Env C = make_env(w, e, act, obs, rew, term); run_env_step(C, w->team, 0); }
}
void dge_reset(EmulWorld* w, const uint8_t* mask, float* obs, float* rew, uint8_t* term) {
  for (int e = 0; e < w->n_envs; e++) { if (mask && !mask[e]) continue; poison(w); Env C = make_env(w, e, nullptr, obs, rew, term); run_env_reset(C, w->team, 0); }
}
void dge_observe(EmulWorld* w, float* obs, float* rew, uint8_t* term) {
  for (int e = 0; e < w->n_envs; e++) { poison(w); Env C = make_env(w, e, nullptr, obs, rew, term); run_env_observe(C, w->team, 0); }
}
unsigned dge_contacts_dropped(EmulWorld* w) { return w->dropped; }
// physics only (no add-on ops): nsub = 0 refreshes the link cache
void dge_physics(EmulWorld* w, int nsub) {
  std::vector<float> o(w->hs.dev.n_obs + 1), r(w->hs.dev.n_rew + 1); std::vector<uint8_t> t(w->hs.dev.n_term + 1);
  for (int e = 0; e < w->n_envs; e++) { Env C = make_env(w, 0, nullptr, o.data(), r.data(), t.data()); C.st = w->state.data() + (size_t)e * w->hs.dev.S; C.pr = w->param.data() + (size_t)e * w->hs.dev.P; run_physics(C, w->team, nsub, nsub > 0, 0); }
}

// The kernels that read state rows, on explicit rows: state [n_envs][S], param [n_envs][P], obs [n_envs][n_obs].
// dg_ray_kernel: the ray_sensor ops; mask (one byte per environment, null: all): only those environments are cast.
void dge_rays(EmulWorld* w, const float* state, float* obs, int n_envs, const uint8_t* mask) {
  const DevScene& d = w->hs.dev;
  std::vector<float> mov((size_t)d.nshw * 12 + 1);
  for (int e = 0; e < n_envs; e++) {
    if (mask && !mask[e]) continue;
    Env C = row_env(d, const_cast<float*>(state) + (size_t)e * d.S);
    C.obs = obs + (size_t)e * d.n_obs;
    ray_stage_shapes(C, mov.data(), 0, 1);
    ray_env(C, mov.data(), 0, 1);
  }
}
// dg_dyn_kernel, with the arguments of dg_body_dynamics (validated by the caller)
void dge_dynamics(EmulWorld* w, int body, int link, const float* point, const float* q, const float* qd, const float* qdd,
                  float* jac, float* mass, float* tau, const float* state, const float* param, int n_envs) {
  const DevScene& d = w->hs.dev;
  const DynArgs a = dyn_args(d, body, link, point, q, qd, qdd, jac, mass, tau);
  std::vector<unsigned long long> msk(a.nl);
  std::vector<float> L((size_t)DL_W_ * a.nl), col((size_t)DC_W_ * a.n + 1), pt(4);
  for (int e = 0; e < n_envs; e++) {
    const float* pr = param + (size_t)e * d.P;
    dyn_chain(d, a, state + (size_t)e * d.S, pr, e, msk.data(), L.data(), col.data());
    dyn_links(d, a, pr, L.data(), pt.data(), 0, 1);
    dyn_outputs(a, e, msk.data(), L.data(), col.data(), pt.data(), 0, 1);
  }
}
// dg_ik_kernel, with the arguments of dg_body_ik (validated by the caller; link is the body's link index)
void dge_ik(EmulWorld* w, int body, int link, const float* tpos, const float* torn, const float* q0, const float* lim, int iters,
            float threshold, float* q_out, float* err, const float* state, int n_envs) {
  DevScene d = w->hs.dev;
  const int* bi = d.body_i + DG_BODY_I_W * body;
  IkArgs a = ik_args(d, bi, body, link, tpos, torn, q0, lim, iters, threshold, q_out, err);
  std::vector<float> rec((size_t)n_envs * a.rec_stride);
  a.rec = rec.data();
  ik_variant(bi[4], a.use_orn, [&](auto maxd, auto m) { ik_solve_all<decltype(maxd)::value, decltype(m)::value>(d, a, state, n_envs); });
}
}
