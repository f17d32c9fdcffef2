// tests/emul/ik_emul.cpp - TEST INFRASTRUCTURE: compiles the inverse-kinematics query (csrc/dg_ik.cuh over the step kernel's IK
// routines in csrc/dg_env.cuh) with g++, so that the fp32 arithmetic of dg_ik_kernel can be checked against the fp64 reference
// (tests/ik_reference.py) without a GPU.  Every environment is solved in turn, as one lane of the kernel solves it.  Never
// shipped, never used by the product path.
#include <stdint.h>
#include <stdio.h>

#include <vector>

#include "../../diy_gym_b200/csrc/dg_ik.cuh"

using namespace dg;

struct IkWorld { HostScene hs; };

template <int MAXD, int M>
static void solve_all(const DevScene& d, const IkArgs& a, const float* state, int n_envs) {
  std::vector<float> scr(IkFastScratch<MAXD>::floats);
  for (int e = 0; e < n_envs; e++) {
    Env C;
    C.sc = &d; C.link_i = d.link_i; C.link_f = d.link_f; C.link_x = d.link_x; C.st = a.rec + (size_t)e * a.rec_stride;
    ik_env<MAXD, M>(C, a, state + (size_t)e * d.S, e, scr.data());
  }
}

extern "C" {
// team: the team size of the emulated step world (scenes with welds need the row-space solver of a team of several lanes)
IkWorld* dgi_create(const int32_t* ibuf, int ni, const double* fbuf, int nf, int team) {
  IkWorld* w = new IkWorld();
  if (!w->hs.build(ibuf, ni, fbuf, nf, team, 2)) { fprintf(stderr, "ik_emul: %s\n", w->hs.error.c_str()); delete w; return nullptr; }
  return w;
}
void dgi_destroy(IkWorld* w) { delete w; }
// The arguments of dg_body_ik (validated by the caller; link is the body's link index), with host state rows [n_envs][S].
void dgi_ik(IkWorld* w, int body, int link, const float* tpos, const float* torn, const float* q0, const float* lim, int iters,
            float threshold, float* q_out, float* err, const float* state, int n_envs) {
  DevScene d = w->hs.dev;
  const int* bi = d.body_i + DG_BODY_I_W * body;
  const int ndb = bi[4];
  IkArgs a;
  a.body = body; a.link = bi[1] + link; a.use_orn = torn != nullptr;
  a.s_q = DG_SO(&d, S_Q); a.s_bpos = DG_SO(&d, S_BPOS); a.s_bquat = DG_SO(&d, S_BQUAT);
  a.seed_floats = ik_scene(d, iters, threshold);
  a.rec_stride = a.seed_floats + d.ik_stride;
  a.tpos = tpos; a.torn = torn; a.q0 = q0; a.lim = lim; a.q_out = q_out; a.err = err;
  std::vector<float> rec((size_t)n_envs * a.rec_stride);
  a.rec = rec.data();
  if (ndb <= 6) { if (a.use_orn) solve_all<6, 6>(d, a, state, n_envs); else solve_all<6, 3>(d, a, state, n_envs); }
  else if (ndb <= 12) { if (a.use_orn) solve_all<12, 6>(d, a, state, n_envs); else solve_all<12, 3>(d, a, state, n_envs); }
  else solve_all<0, 0>(d, a, state, n_envs);
}
}
