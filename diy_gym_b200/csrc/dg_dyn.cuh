// dg_dyn.cuh - rigid-body dynamics queries of one body (pybullet's calculateJacobian / calculateMassMatrix /
// calculateInverseDynamics), evaluated per environment from the state and parameter rows by dg_dyn_kernel (dg_kernels.cu).
//
// Generalized velocity nu of a body: floating base (kind 2) [omega_base (world), v_base (world, base COM), qd (its DoF in order)],
// fixed base qd only; n = len(nu).  Every quantity below is in world axes.  Column c of the Jacobian of a point P of link k is
//   Jw = w_c,  Jv = w_c x (P - o_c) + u_c          when the DoF of column c moves link k (bit c of the link's column mask), else 0
// with  revolute: w = joint axis, o = a point on it, u = 0;  prismatic: w = 0, u = axis;  base omega_i: w = e_i, o = base COM;
// base v_i: u = e_i.  Then, summing over every link k of the body (the base included when it floats):
//   M_ij  = sum_k m_k Jv_ki . Jv_kj + w_i^T I_k w_j                     (k moved by both i and j)
//   tau_i = sum_k Jv_ki . f_k + w_i . n_k,   f_k = m_k (a_k - g),  n_k = I_k alpha_k + omega_k x I_k omega_k
// where a_k / alpha_k are the link's COM / angular accelerations at (q, nu, nu_dot = qdd) from one forward pass (recursive
// Newton-Euler in world axes: tau = M qdd + C nu + G without forming M).  Masses and principal inertias come from the parameter
// row (P_MASS, P_INERTIA: dynamics_randomizer is honoured); joint damping, motors, limits, contacts and welds are not included.
//
// The routines are DG_FN so that the test-only CPU build (tests/emul/dyn_emul.cpp) runs the same fp32 arithmetic as the kernel.
// One environment is evaluated in three phases: dyn_chain (one lane: the sequential pass over the links), dyn_links (lanes over
// links: world inertias and the link wrenches), dyn_outputs (lanes over columns / matrix entries); a barrier between phases.
#pragma once
#include "dg_math.cuh"
#include "dg_scene.h"

namespace dg {

// largest n the queries accept (bit c of a 64-bit mask marks the links that DoF c moves)
enum { DG_DYN_MAXN = 64 };   // (= DG_DYN_MAX_N of include/diygym_b200.h)
// per-link record in the scratch (floats): COM c, wrench f / n, world inertia (xx yy zz xy xz yz), mass, rotation, angular /
// linear velocity, angular / linear acceleration
enum { DL_C = 0, DL_F = 3, DL_N = 6, DL_I = 9, DL_M = 15, DL_R = 16, DL_W = 25, DL_V = 28, DL_AL = 31, DL_A = 34, DL_W_ = 40 };
// per-column record: w (3), u (3), o (3)
enum { DC_W = 0, DC_U = 3, DC_O = 6, DC_W_ = 9 };

struct DynArgs {
  int body, link, n, nl;            // body, link (-1: base), generalized coordinates, link records (links of the body + 1)
  float point[3];                   // point of the Jacobian, in the link's COM frame
  const float *q, *qd, *qdd;        // [N][nd], [N][n], [N][n]; null: state row, state row, zero
  float *jac, *mass, *tau;          // [N][6][n] (linear rows first), [N][n][n], [N][n]; null: not computed
};

// scratch of one environment: nl 64-bit column masks, then nl link records, n column records and the point (floats)
DG_HD int dyn_scratch_floats(int nl, int n) { return (2 * nl + DL_W_ * nl + DC_W_ * n + 4 + 3) & ~3; }

DG_HD void dyn_cross_add(float* o, const float* a, const float* b) {   // o += a x b
  float t[3]; v_cross(t, a, b); v_add(o, o, t);
}

// Sequential pass (one lane): link poses from q, joint columns, velocities and accelerations, base first.  st / pr: the
// environment's state and parameter rows; e: its index in the q / qd / qdd inputs.
DG_FN void dyn_chain(const DevScene& sc, const DynArgs& a, const float* st, const float* pr, int e, unsigned long long* msk, float* L, float* col) {
  const int* bi = sc.body_i + DG_BODY_I_W * a.body;
  const int kind = bi[0], l0 = bi[1], nlb = bi[2], d0 = bi[3], fb = kind == 2 ? 6 : 0;
  const float* q = a.q ? a.q + (size_t)e * (a.n - fb) : nullptr;
  const float* qd = a.qd ? a.qd + (size_t)e * a.n : nullptr;
  const float* qdd = a.qdd ? a.qdd + (size_t)e * a.n : nullptr;
  const float* sq = st + DG_SO(&sc, S_Q); const float* sqd = st + DG_SO(&sc, S_QD);
  float* B = L;
  q_to_mat(B + DL_R, st + DG_SO(&sc, S_BQUAT) + 4 * a.body); v_cpy(B + DL_C, st + DG_SO(&sc, S_BPOS) + 3 * a.body);
  for (int i = 0; i < 3; i++) { B[DL_W + i] = 0.f; B[DL_V + i] = 0.f; B[DL_AL + i] = 0.f; B[DL_A + i] = 0.f; }
  B[DL_M] = 0.f; msk[0] = 0ull;
  if (kind == 2) {
    for (int i = 0; i < 3; i++) {
      B[DL_W + i] = qd ? qd[i] : st[DG_SO(&sc, S_BOMEGA) + 3 * a.body + i];
      B[DL_V + i] = qd ? qd[3 + i] : st[DG_SO(&sc, S_BVEL) + 3 * a.body + i];
      if (qdd) { B[DL_AL + i] = qdd[i]; B[DL_A + i] = qdd[3 + i]; }
    }
    B[DL_M] = pr[DG_PO(&sc, P_MASS) + a.body];
    msk[0] = 0x3full;
    for (int i = 0; i < 6; i++) {
      float* cc = col + DC_W_ * i;
      for (int k = 0; k < 9; k++) cc[k] = 0.f;
      if (i < 3) { cc[DC_W + i] = 1.f; v_cpy(cc + DC_O, B + DL_C); } else cc[DC_U + i - 3] = 1.f;
    }
  }
  for (int k = 0; k < nlb; k++) {
    const int gl = l0 + k; const int* li = sc.link_i + DG_LINK_I_W * gl; const float* lf = sc.link_f + DG_LINK_F_W * gl;
    const float* R0 = sc.link_x + 16 * gl;
    const float* P = L + DL_W_ * (li[1] < 0 ? 0 : li[1] - l0 + 1);
    float* K = L + DL_W_ * (k + 1);
    const int jt = li[2], dof = li[3], c = dof >= 0 ? fb + dof - d0 : -1;
    const float qk = dof < 0 ? 0.f : (q ? q[dof - d0] : sq[dof]);
    const float qdk = dof < 0 ? 0.f : (qd ? qd[c] : sqd[dof]);
    const float qddk = dof < 0 || !qdd ? 0.f : qdd[c];
    // joint transform (compiler/scene.py): child rotation R0 Rot(a, q) / R0, child COM e + Rrel d / e + R0 (d + a q) in the parent's COM frame
    float Rrel[9], r[3], t[3];
    if (jt == 1) { float Ra[9]; axis_angle_mat(Ra, lf + 10, qk, true); m_mul(Rrel, R0, Ra); m_vec(t, Rrel, lf + 7); }
    else if (jt == 2) { m_cpy(Rrel, R0); const float dd[3] = {lf[7] + lf[10] * qk, lf[8] + lf[11] * qk, lf[9] + lf[12] * qk}; m_vec(t, R0, dd); }
    else { m_cpy(Rrel, R0); m_vec(t, R0, lf + 7); }
    v_add(r, lf + 4, t);
    m_mul(K + DL_R, P + DL_R, Rrel);
    m_vec(t, P + DL_R, r); v_add(K + DL_C, P + DL_C, t);
    float s[3], o[3], rho[3];
    m_vec(s, K + DL_R, lf + 10); m_vec(t, K + DL_R, lf + 7); v_sub(o, K + DL_C, t);
    v_sub(rho, K + DL_C, P + DL_C);
    // rigid motion with the parent, then the joint's own contribution
    const float *wp = P + DL_W, *alp = P + DL_AL;
    float *wk = K + DL_W, *vk = K + DL_V, *alk = K + DL_AL, *ak = K + DL_A;
    v_cpy(wk, wp); v_cpy(alk, alp);
    v_cpy(vk, P + DL_V); dyn_cross_add(vk, wp, rho);
    if (jt == 1) {
      // a_k = a_o + alpha_k x (c_k - o) + omega_k x (omega_k x (c_k - o)), o on the axis (fixed in parent and child)
      float sq_[3], po[3], ro[3], wxr[3];
      v_scale(sq_, s, qdk);
      v_add(wk, wk, sq_); dyn_cross_add(alk, wp, sq_); v_madd(alk, s, qddk);
      v_sub(ro, K + DL_C, o); dyn_cross_add(vk, sq_, ro);
      v_sub(po, o, P + DL_C);
      v_cpy(ak, P + DL_A); dyn_cross_add(ak, alp, po); v_cross(wxr, wp, po); dyn_cross_add(ak, wp, wxr);
      dyn_cross_add(ak, alk, ro); v_cross(wxr, wk, ro); dyn_cross_add(ak, wk, wxr);
    } else {
      float wxr[3];
      v_cpy(ak, P + DL_A); dyn_cross_add(ak, alp, rho); v_cross(wxr, wp, rho); dyn_cross_add(ak, wp, wxr);
      if (jt == 2) {   // sliding along s: relative velocity qd s, Coriolis 2 omega_p x qd s, relative acceleration qdd s
        v_madd(vk, s, qdk); float sq_[3]; v_scale(sq_, s, 2.f * qdk); dyn_cross_add(ak, wp, sq_); v_madd(ak, s, qddk);
      }
    }
    K[DL_M] = pr[DG_PO(&sc, P_MASS) + sc.nb + gl];
    msk[k + 1] = msk[li[1] < 0 ? 0 : li[1] - l0 + 1] | (c >= 0 ? 1ull << c : 0ull);
    if (c >= 0) {
      float* cc = col + DC_W_ * c;
      for (int i = 0; i < 3; i++) { cc[DC_W + i] = jt == 1 ? s[i] : 0.f; cc[DC_U + i] = jt == 2 ? s[i] : 0.f; cc[DC_O + i] = o[i]; }
    }
  }
}

// Lanes over links: world inertia R diag(I) R^T, f = m (a - g), n = I alpha + omega x I omega; lane 0 also places the point.
DG_FN void dyn_links(const DevScene& sc, const DynArgs& a, const float* pr, float* L, float* pt, int ln, int nt) {
  const int* bi = sc.body_i + DG_BODY_I_W * a.body;
  for (int k = ln; k < a.nl; k += nt) {
    float* K = L + DL_W_ * k;
    const int f = k == 0 ? a.body : sc.nb + bi[1] + k - 1;
    const float* Id = pr + DG_PO(&sc, P_INERTIA) + 3 * f; const float* R = K + DL_R;
    float* Iw = K + DL_I;
    Iw[0] = R[0] * R[0] * Id[0] + R[1] * R[1] * Id[1] + R[2] * R[2] * Id[2];
    Iw[1] = R[3] * R[3] * Id[0] + R[4] * R[4] * Id[1] + R[5] * R[5] * Id[2];
    Iw[2] = R[6] * R[6] * Id[0] + R[7] * R[7] * Id[1] + R[8] * R[8] * Id[2];
    Iw[3] = R[0] * R[3] * Id[0] + R[1] * R[4] * Id[1] + R[2] * R[5] * Id[2];
    Iw[4] = R[0] * R[6] * Id[0] + R[1] * R[7] * Id[1] + R[2] * R[8] * Id[2];
    Iw[5] = R[3] * R[6] * Id[0] + R[4] * R[7] * Id[1] + R[5] * R[8] * Id[2];
    const float m = K[DL_M], *w = K + DL_W, *al = K + DL_AL;
    for (int i = 0; i < 3; i++) K[DL_F + i] = m * (K[DL_A + i] - sc.g[i]);
    const float Iwv[3] = {Iw[0] * w[0] + Iw[3] * w[1] + Iw[4] * w[2], Iw[3] * w[0] + Iw[1] * w[1] + Iw[5] * w[2], Iw[4] * w[0] + Iw[5] * w[1] + Iw[2] * w[2]};
    float* nn = K + DL_N;
    nn[0] = Iw[0] * al[0] + Iw[3] * al[1] + Iw[4] * al[2]; nn[1] = Iw[3] * al[0] + Iw[1] * al[1] + Iw[5] * al[2]; nn[2] = Iw[4] * al[0] + Iw[5] * al[1] + Iw[2] * al[2];
    dyn_cross_add(nn, w, Iwv);
  }
  if (ln == 0) { const float* K = L + DL_W_ * (a.link + 1); float t[3]; m_vec(t, K + DL_R, a.point); v_add(pt, K + DL_C, t); }
}

// Jv of column c at point p (w x (p - o) + u)
DG_HD void dyn_jv(float* jv, const float* cc, const float* p) { float r[3]; v_sub(r, p, cc + DC_O); v_cross(jv, cc + DC_W, r); v_add(jv, jv, cc + DC_U); }

// Lanes over Jacobian columns, upper-triangle entries of M (mirrored) and generalized forces.  e: environment index of the outputs.
DG_FN void dyn_outputs(const DynArgs& a, int e, const unsigned long long* msk, const float* L, const float* col, const float* pt, int ln, int nt) {
  const int n = a.n;
  if (a.jac) {
    float* J = a.jac + (size_t)e * 6 * n;
    const unsigned long long lm = msk[a.link + 1];
    for (int c = ln; c < n; c += nt) {
      const float* cc = col + DC_W_ * c; float jv[3] = {0.f, 0.f, 0.f}, jw[3] = {0.f, 0.f, 0.f};
      if ((lm >> c) & 1ull) { dyn_jv(jv, cc, pt); v_cpy(jw, cc + DC_W); }
      for (int r = 0; r < 3; r++) { J[r * n + c] = jv[r]; J[(3 + r) * n + c] = jw[r]; }
    }
  }
  if (a.mass) {
    float* M = a.mass + (size_t)e * n * n;
    const int np = n * (n + 1) / 2;
    for (int p = ln; p < np; p += nt) {
      int i = 0, j = p;
      while (j >= n - i) { j -= n - i; i++; }
      j += i;
      const float *ci = col + DC_W_ * i, *cj = col + DC_W_ * j;
      const unsigned long long both = (1ull << i) | (1ull << j);
      float s = 0.f;
      for (int k = 0; k < a.nl; k++) {
        if ((msk[k] & both) != both) continue;
        const float* K = L + DL_W_ * k; const float* I = K + DL_I;
        float vi[3], vj[3];
        dyn_jv(vi, ci, K + DL_C); dyn_jv(vj, cj, K + DL_C);
        const float* wj = cj + DC_W;
        const float Iwj[3] = {I[0] * wj[0] + I[3] * wj[1] + I[4] * wj[2], I[3] * wj[0] + I[1] * wj[1] + I[5] * wj[2], I[4] * wj[0] + I[5] * wj[1] + I[2] * wj[2]};
        s += K[DL_M] * v_dot(vi, vj) + v_dot(ci + DC_W, Iwj);
      }
      M[i * n + j] = s; M[j * n + i] = s;
    }
  }
  if (a.tau) {
    float* T = a.tau + (size_t)e * n;
    for (int c = ln; c < n; c += nt) {
      const float* cc = col + DC_W_ * c; float s = 0.f;
      for (int k = 0; k < a.nl; k++) {
        if (!((msk[k] >> c) & 1ull)) continue;
        const float* K = L + DL_W_ * k; float jv[3];
        dyn_jv(jv, cc, K + DL_C);
        s += v_dot(jv, K + DL_F) + v_dot(cc + DC_W, K + DL_N);
      }
      T[c] = s;
    }
  }
}

}  // namespace dg
