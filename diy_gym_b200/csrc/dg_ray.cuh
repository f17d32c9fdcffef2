// dg_ray.cuh - rays against shapes: the per-ray routines shared by the camera (visual shapes, dg_render_kernel) and the
// ray_sensor add-on (collision shapes, dg_ray_kernel), and the per-environment evaluation of the ray_sensor ops.
//
// The routines are DG_HD so that the test-only CPU emulation (tests/emul) runs the same fp32 arithmetic as the kernel.
#pragma once
#include "dg_env.cuh"

namespace dg {

// nearest hit of a ray (shape-local origin o, direction dir) within (1e-9, tmax)
DG_HD bool ray_shape(int type, const float* d, const float* o, const float* dir, float tmax, float* t_out, float* n_out) {
  float best = tmax; bool hit = false; float nb_[3] = {0, 0, 1};
  if (type == SHAPE_SPHERE || type == SHAPE_CAPSULE) {
    int nsph = type == SHAPE_SPHERE ? 1 : 2;
    for (int s = 0; s < nsph; s++) {
      float cz = type == SHAPE_SPHERE ? 0.f : (s ? d[1] : -d[1]);
      float oc[3] = {o[0], o[1], o[2] - cz};
      float A = v_dot(dir, dir), B = v_dot(oc, dir), Cc = v_dot(oc, oc) - d[0] * d[0], disc = B * B - A * Cc;
      if (disc < 0) continue;
      float t = (-B - sqrtf(disc)) / A;
      if (t > 1e-9f && t < best) { best = t; hit = true; for (int i = 0; i < 3; i++) nb_[i] = (oc[i] + t * dir[i]) / d[0]; }
    }
  }
  if (type == SHAPE_CAPSULE || type == SHAPE_CYLINDER) {
    float A = dir[0] * dir[0] + dir[1] * dir[1], B = o[0] * dir[0] + o[1] * dir[1], Cc = o[0] * o[0] + o[1] * o[1] - d[0] * d[0];
    float disc = B * B - A * Cc;
    if (A > 1e-18f && disc >= 0) {
      float t = (-B - sqrtf(disc)) / A, z = o[2] + t * dir[2];
      if (t > 1e-9f && t < best && fabsf(z) <= d[1]) { best = t; hit = true; nb_[0] = (o[0] + t * dir[0]) / d[0]; nb_[1] = (o[1] + t * dir[1]) / d[0]; nb_[2] = 0; }
    }
    if (type == SHAPE_CYLINDER && fabsf(dir[2]) > 1e-18f) for (int s = -1; s <= 1; s += 2) {
      float t = (s * d[1] - o[2]) / dir[2], x = o[0] + t * dir[0], y = o[1] + t * dir[1];
      if (t > 1e-9f && t < best && x * x + y * y <= d[0] * d[0]) { best = t; hit = true; nb_[0] = 0; nb_[1] = 0; nb_[2] = (float)s; }
    }
  }
  if (type == SHAPE_BOX) {
    // slab test without branches: the three axes are independent (reciprocals by the SFU, ~1 ulp: the depth tolerance
    // is 1e-4); a ray parallel to a slab gets (-inf, +inf) inside it and an empty interval outside
    float t0 = -1e30f, t1 = 1e30f; int ax0 = 0; float sg0 = 1;
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const bool par = fabsf(dir[i]) < 1e-18f, inside = fabsf(o[i]) <= d[i];
#if defined(__CUDA_ARCH__)
      const float inv = __fdividef(1.0f, par ? 1.0f : dir[i]);
#else
      const float inv = 1.0f / (par ? 1.0f : dir[i]);
#endif
      const float ua = (-d[i] - o[i]) * inv, ub = (d[i] - o[i]) * inv;
      float ta = fminf(ua, ub), tb = fmaxf(ua, ub); const float sg = ua > ub ? 1.f : -1.f;
      ta = par ? (inside ? -1e30f : 1e30f) : ta; tb = par ? (inside ? 1e30f : -1e30f) : tb;
      if (ta > t0) { t0 = ta; ax0 = i; sg0 = sg; }
      t1 = fminf(t1, tb);
    }
    if (t0 <= t1 && t0 > 1e-9f && t0 < best) { best = t0; hit = true; nb_[0] = ax0 == 0 ? sg0 : 0.f; nb_[1] = ax0 == 1 ? sg0 : 0.f; nb_[2] = ax0 == 2 ? sg0 : 0.f; }
  }
  if (hit) { *t_out = best; v_cpy(n_out, nb_); }
  return hit;
}

// ---------------------------------------------------------------- ray_sensor ----------------------------------------
// Op RAY_SENSOR (addons/builtin.py RaySensor): iargs [frame (-1: the world), R, flags (1: hit object ids)], fargs [xyz (3),
// quat (4), min, max, R unit directions in the sensor frame (3 each)].  Observation: R distances, then (flags & 1) R body ids.
// The op code (compiler/scene.py KERNEL_OPS): the step kernel does not know it and skips the op.
#define OP_RAY_SENSOR 19
enum { RAY_FA_XYZ = 0, RAY_FA_QUAT = 3, RAY_FA_MIN = 7, RAY_FA_MAX = 8, RAY_FA_DIRS = 9 };

// Origin (shape-local o) inside the shape: the ray then does not report it (only entry surfaces count).  `planes` / np_: the
// reduced convex hull of a mesh shape, which replaces the fitted primitive when np_ > 0 (outward unit normals n, offsets:
// n . x <= offset inside).
DG_HD bool ray_inside(int type, const float* d, const float* planes, int np_, const float* o) {
  if (np_ > 0) {
    for (int k = 0; k < np_; k++) { const float* q = planes + 4 * k; if (v_dot(q, o) - q[3] > 0.f) return false; }
    return true;
  }
  if (type == SHAPE_SPHERE) return v_dot(o, o) <= d[0] * d[0];
  if (type == SHAPE_BOX) return fabsf(o[0]) <= d[0] && fabsf(o[1]) <= d[1] && fabsf(o[2]) <= d[2];
  const float r2 = o[0] * o[0] + o[1] * o[1];
  if (type == SHAPE_CYLINDER) return r2 <= d[0] * d[0] && fabsf(o[2]) <= d[1];
  const float z = fminf(fmaxf(o[2], -d[1]), d[1]), dz = o[2] - z;   // capsule: distance to the axis segment
  return r2 + dz * dz <= d[0] * d[0];
}

// Nearest entry of a ray into a convex hull within (1e-9, tmax): Cyrus-Beck clip of the ray against the hull's planes.
DG_HD bool ray_hull(const float* planes, int np_, const float* o, const float* dir, float tmax, float* t_out) {
  float te = -1e30f, tx = tmax;
  for (int k = 0; k < np_; k++) {
    const float* q = planes + 4 * k;
    const float num = q[3] - v_dot(q, o), den = v_dot(q, dir);   // num >= 0: the origin is on the inner side of this plane
    if (fabsf(den) < 1e-18f) { if (num < 0.f) return false; continue; }
    const float t = num / den;
    if (den < 0.f) te = fmaxf(te, t); else tx = fminf(tx, t);
  }
  if (te <= tx && te > 1e-9f && te < tmax) { *t_out = te; return true; }
  return false;
}

// World pose (R 9, p 3) of a collision shape that is not baked: from the COM-frame pose in the state row's link cache.
DG_HD void ray_shape_world(const Env& C, int s, float* out) {
  const float* sf = C.sc->shape_f + DG_SHAPE_F_W * s;
  float p[3], q[4], v[3], w[3], R[9], Rs[9], t[3];
  frame_com_state(C, C.sc->shape_i[DG_SHAPE_I_W * s + 1], p, q, v, w); q_to_mat(R, q); q_to_mat(Rs, sf + 3); m_mul(out, R, Rs);
  m_vec(t, R, sf); v_add(out + 9, p, t);
}

// Nearest hit of the world ray org + t dir, t in (tmin, tmax], over every collision shape of the scene.  mov: world poses of the
// non-baked shapes [DevScene::shape_slot][12]; baked ones come from DevScene::shape_wb.  Returns the distance (tmax on a miss) and
// the body index of the shape hit (-1 on a miss).
DG_HD float ray_cast(const DevScene& sc, const float* mov, const float* org, const float* dir, float tmin, float tmax, int* body) {
  float best = tmax - tmin; int hb = -1;   // ray parameter from the point at tmin
  for (int s = 0; s < sc.ns; s++) {
    const int* si = sc.shape_i + DG_SHAPE_I_W * s; const float* sf = sc.shape_f + DG_SHAPE_F_W * s;
    const int slot = sc.shape_slot[s];
    const float* P = slot >= 0 ? mov + 12 * slot : sc.shape_wb + 12 * s;
    // bounding sphere: skip the shape when the ray's line misses it or when it lies wholly before tmin or beyond the best hit
    float oc[3]; v_sub(oc, org, P + 9);
    const float r = sf[11], b = v_dot(oc, dir), c = v_dot(oc, oc) - r * r;
    if (b * b < c || -b - r > tmin + best || -b + r < tmin) continue;
    float ol[3], dl[3], om[3];
    mT_vec(ol, P, oc); mT_vec(dl, P, dir);
    om[0] = fmaf(tmin, dl[0], ol[0]); om[1] = fmaf(tmin, dl[1], ol[1]); om[2] = fmaf(tmin, dl[2], ol[2]);
    const int np_ = si[5] > 0 ? si[7] : 0; const float* planes = sc.hull_f + si[6];
    if (ray_inside(si[2], sf + 7, planes, np_, om)) continue;
    float t, nn[3];
    const bool hit = np_ > 0 ? ray_hull(planes, np_, om, dl, best, &t) : ray_shape(si[2], sf + 7, om, dl, best, &t, nn);
    if (hit) { best = t; hb = si[0]; }
  }
  *body = hb;
  return hb >= 0 ? tmin + best : tmax;
}

// World poses of the non-baked shapes of one environment into mov [DevScene::nshw][12], lane `ln` of `nt`.
DG_HD void ray_stage_shapes(const Env& C, float* mov, int ln, int nt) {
  const DevScene& sc = *C.sc;
  for (int s = ln; s < sc.ns; s += nt) { const int slot = sc.shape_slot[s]; if (slot >= 0) ray_shape_world(C, s, mov + 12 * slot); }
}
// Every ray_sensor op of one environment: lane `ln` of `nt` takes rays ln, ln + nt, ...  mov must hold the poses of the
// non-baked shapes (ray_stage_shapes, then a barrier of the nt lanes).  Other ops are skipped.
DG_HD void ray_env(const Env& C, const float* mov, int ln, int nt) {
  const DevScene& sc = *C.sc;
  for (int k = 0; k < sc.nop; k++) {
    const int* op = sc.op_i + DG_OP_I_W * k;
    if (op[0] != OP_RAY_SENSOR) continue;
    const int* ia = sc.oparg_i + op[1]; const float* fa = sc.oparg_f + op[2];
    const int nr = ia[1]; float* o = C.obs + op[4];
    // sensor pose: the frame's URDF link pose (the camera's convention), then xyz / quat in that frame
    float Rp[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, pp[3] = {0, 0, 0}, Rl[9], Rs[9], ps[3], t[3];
    if (ia[0] >= 0) { float q[4]; frame_link_pose(C, ia[0], pp, q); q_to_mat(Rp, q); }
    q_to_mat(Rl, fa + RAY_FA_QUAT); m_mul(Rs, Rp, Rl); m_vec(t, Rp, fa + RAY_FA_XYZ); v_add(ps, pp, t);
    const float tmin = fa[RAY_FA_MIN], tmax = fa[RAY_FA_MAX];
    for (int r = ln; r < nr; r += nt) {
      float dw[3]; int hb;
      m_vec(dw, Rs, fa + RAY_FA_DIRS + 3 * r);
      o[r] = ray_cast(sc, mov, ps, dw, tmin, tmax, &hb);
      if (ia[2] & 1) o[nr + r] = (float)hb;
    }
  }
}

}  // namespace dg
