// tests/emul/ray_emul.cpp - TEST INFRASTRUCTURE: compiles the ray_sensor routines of csrc/dg_ray.cuh with g++, so that the fp32
// arithmetic of dg_ray_kernel can be checked against the fp64 reference (tests/ray_reference.py) without a GPU.  It casts the rays
// of every ray_sensor op from state rows as they are, one lane per environment, as the kernel does after every step / reset /
// observe launch.  Never shipped, never used by the product path.
#include <stdint.h>
#include <stdio.h>

#include <vector>

#include "../../diy_gym_b200/csrc/dg_ray.cuh"

using namespace dg;

struct RayWorld { HostScene hs; };

extern "C" {
RayWorld* dgr_create(const int32_t* ibuf, int ni, const double* fbuf, int nf) {
  RayWorld* w = new RayWorld();
  if (!w->hs.build(ibuf, ni, fbuf, nf, 1, 2)) { fprintf(stderr, "ray_emul: %s\n", w->hs.error.c_str()); delete w; return nullptr; }
  return w;
}
void dgr_destroy(RayWorld* w) { delete w; }
// state [n_envs][S], obs [n_envs][n_obs]; mask (one byte per environment, null: all): only those environments are cast
void dgr_rays(RayWorld* w, float* state, float* obs, int n_envs, const uint8_t* mask) {
  const DevScene& d = w->hs.dev;
  std::vector<float> mov((size_t)d.nshw * 12 + 1);
  for (int e = 0; e < n_envs; e++) {
    if (mask && !mask[e]) continue;
    Env C; C.sc = &d; C.st = state + (size_t)e * d.S; C.obs = obs + (size_t)e * d.n_obs;
    C.ws = nullptr; C.wg = nullptr; C.pr = nullptr; C.dbg = nullptr; C.dropped = nullptr; C.rs_used = nullptr; C.no_hot = 0;
    C.link_i = d.link_i; C.link_f = d.link_f; C.link_x = d.link_x;
    ray_stage_shapes(C, mov.data(), 0, 1);
    ray_env(C, mov.data(), 0, 1);
  }
}
}
