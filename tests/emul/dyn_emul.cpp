// tests/emul/dyn_emul.cpp - TEST INFRASTRUCTURE: compiles the dynamics-query routines of csrc/dg_dyn.cuh with g++, so that the
// fp32 arithmetic of dg_dyn_kernel can be checked against the fp64 reference (tests/dynamics_reference.py) without a GPU.  It runs
// the kernel's three phases for every environment, one lane each.  Never shipped, never used by the product path.
#include <stdint.h>
#include <stdio.h>

#include <vector>

#include "../../diy_gym_b200/csrc/dg_dyn.cuh"

using namespace dg;

struct DynWorld { HostScene hs; };

extern "C" {
DynWorld* dgd_create(const int32_t* ibuf, int ni, const double* fbuf, int nf) {
  DynWorld* w = new DynWorld();
  if (!w->hs.build(ibuf, ni, fbuf, nf, 1, 2)) { fprintf(stderr, "dyn_emul: %s\n", w->hs.error.c_str()); delete w; return nullptr; }
  return w;
}
void dgd_destroy(DynWorld* w) { delete w; }
// The arguments of dg_body_dynamics (validated by the caller), with host state [n_envs][S] and param [n_envs][P] rows.
void dgd_dynamics(DynWorld* w, int body, int link, const float* point, const float* q, const float* qd, const float* qdd,
                  float* jac, float* mass, float* tau, const float* state, const float* param, int n_envs) {
  const DevScene& d = w->hs.dev;
  const int* bi = d.body_i + DG_BODY_I_W * body;
  DynArgs a;
  a.body = body; a.link = link; a.n = (bi[0] == 2 ? 6 : 0) + bi[4]; a.nl = bi[2] + 1;
  for (int i = 0; i < 3; i++) a.point[i] = point[i];
  a.q = q; a.qd = qd; a.qdd = qdd; a.jac = jac; a.mass = mass; a.tau = tau;
  std::vector<unsigned long long> msk(a.nl);
  std::vector<float> L((size_t)DL_W_ * a.nl), col((size_t)DC_W_ * a.n + 1), pt(4);
  for (int e = 0; e < n_envs; e++) {
    const float* pr = param + (size_t)e * d.P;
    dyn_chain(d, a, state + (size_t)e * d.S, pr, e, msk.data(), L.data(), col.data());
    dyn_links(d, a, pr, L.data(), pt.data(), 0, 1);
    dyn_outputs(a, e, msk.data(), L.data(), col.data(), pt.data(), 0, 1);
  }
}
}
