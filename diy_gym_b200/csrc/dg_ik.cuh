// dg_ik.cuh - batched inverse-kinematics query of one body (pybullet's calculateInverseKinematics), one environment per lane
// of dg_ik_kernel (dg_kernels.cu).
//
// The solve is the step kernel's own: ik_solve_fast<MAXD, M> / ik_solve of dg_env.cuh, which the ik_controller op calls.  Those
// routines read the seed q and the base pose through ST(S_Q), ST(S_BPOS) and ST(S_BQUAT), and the iteration count and threshold
// from the scene.  So the kernel runs them on a copy of the DevScene whose state offsets of those three sections point into a
// per-environment seed record [q (sc.nd) | base positions (3 nb) | base quaternions (4 nb)] (ik_scene), and whose ik_iters /
// ik_threshold are the caller's; ik_env fills the record from the caller's seed and the state row before the solve.  Only the
// entries of the queried body are written and read.  Afterwards ik_env evaluates the residual at the returned q with one more
// pass of joint_xform over the chain.
//
// The routines are DG_FN so that the test-only CPU build (tests/emul/emul.cpp) runs the same fp32 arithmetic as the kernel.
#pragma once
#include <type_traits>

#include "dg_env.cuh"

namespace dg {

struct IkArgs {
  int body, link, use_orn;          // body, global index of the target link, 1: the target has an orientation
  int s_q, s_bpos, s_bquat;         // offsets of S_Q / S_BPOS / S_BQUAT in the real state row
  int rec_stride, seed_floats;      // floats per environment in rec; the seed record's share of them (generic scratch after it)
  const float* tpos;                // [N][3] world position of the link frame
  const float* torn;                // [N][4] world orientation (xyzw, any norm) or null
  const float* q0;                  // [N][nd_b] seed or null (the state row's q)
  const float* lim;                 // [N][4][nd_b] lower, upper, range, rest (null-space term) or null
  float* q_out;                     // [N][nd_b]
  float* err;                       // [N][2] position error (m), orientation error angle (rad) at q_out, or null
  float* rec;                       // [N][rec_stride] seed records and generic-path scratch (global memory: ST() assumes it)
};

// floats of the per-thread scratch of ik_solve_fast<MAXD, M>: qb, chain axes and origins, chain, chain position of each DoF
template <int MAXD> struct IkFastScratch { enum { floats = MAXD > 0 ? 2 * MAXD + 7 * DG_MINV_MAXD : 1 }; };

// The scene as the IK routines must see it: S_Q / S_BPOS / S_BQUAT remapped onto the seed record, the caller's iterations and
// threshold.  Returns the record's size in floats.
inline int ik_scene(DevScene& d, int iters, float threshold) {
  DG_SO(&d, S_Q) = 0; DG_SO(&d, S_BPOS) = d.nd; DG_SO(&d, S_BQUAT) = d.nd + 3 * d.nb;
  d.ik_iters = iters; d.ik_threshold = threshold;
  return (d.nd + 7 * d.nb + 3) & ~3;
}

// The arguments of the query of link `link` of `body` (validated by the caller; bi: the body's row of the body table, host memory),
// and d, the copy of the scene the kernel gets, remapped by ik_scene.  The caller points rec at [N][rec_stride] floats.
inline IkArgs ik_args(DevScene& d, const int* bi, int body, int link, const float* tpos, const float* torn, const float* q0,
                      const float* lim, int iters, float threshold, float* q_out, float* err) {
  IkArgs a;
  a.body = body; a.link = bi[1] + link; a.use_orn = torn != nullptr;
  a.s_q = DG_SO(&d, S_Q); a.s_bpos = DG_SO(&d, S_BPOS); a.s_bquat = DG_SO(&d, S_BQUAT);
  a.seed_floats = ik_scene(d, iters, threshold);
  a.rec_stride = a.seed_floats + d.ik_stride;
  a.tpos = tpos; a.torn = torn; a.q0 = q0; a.lim = lim; a.q_out = q_out; a.err = err; a.rec = nullptr;
  return a;
}

// The variant of the solve for a body of ndb DoF (the split of ik_solve_any): ik_solve_fast<MAXD, M> with its arrays in registers up
// to 12 DoF (M = 6 with a target orientation, 3 without), the generic ik_solve (MAXD = M = 0) above.  Calls
// f(std::integral_constant<int, MAXD>(), std::integral_constant<int, M>()).
template <int N> using IkC = std::integral_constant<int, N>;
template <class F> inline void ik_variant(int ndb, bool use_orn, F&& f) {
  if (ndb <= 6) { if (use_orn) f(IkC<6>(), IkC<6>()); else f(IkC<6>(), IkC<3>()); }
  else if (ndb <= 12) { if (use_orn) f(IkC<12>(), IkC<6>()); else f(IkC<12>(), IkC<3>()); }
  else f(IkC<0>(), IkC<0>());
}

// Environment e: fill C.st (the seed record) from the arguments and the state row st, solve, write q_out and err.  MAXD = 0: the
// generic ik_solve (use_orn at run time, M unused), with its scratch behind the seed record; otherwise scr holds
// IkFastScratch<MAXD>::floats floats and M = 3 (position) or 6 (pose).
template <int MAXD, int M>
DG_FN void ik_env(const Env& C, const IkArgs& a, const float* st, int e, float* scr) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * a.body; const int d0 = bi[3], ndb = bi[4];
  float* rec = C.st;
  const float* q0 = a.q0 ? a.q0 + (size_t)e * ndb : st + a.s_q + d0;
  for (int i = 0; i < ndb; i++) ST(S_Q)[d0 + i] = q0[i];
  for (int i = 0; i < 3; i++) ST(S_BPOS)[3 * a.body + i] = st[a.s_bpos + 3 * a.body + i];
  for (int i = 0; i < 4; i++) ST(S_BQUAT)[4 * a.body + i] = st[a.s_bquat + 4 * a.body + i];
  float tpos[3] = {a.tpos[3 * e], a.tpos[3 * e + 1], a.tpos[3 * e + 2]}, torn[4] = {0, 0, 0, 1};
  if (a.use_orn) { for (int i = 0; i < 4; i++) torn[i] = a.torn[4 * (size_t)e + i]; q_norm(torn); }
  const float* lim = a.lim ? a.lim + (size_t)e * 4 * ndb : nullptr;   // null-space term exactly when limits are given
  const float *lo = lim, *up = lim ? lim + ndb : nullptr, *rg = lim ? lim + 2 * ndb : nullptr, *rs = lim ? lim + 3 * ndb : nullptr;
  if constexpr (MAXD > 0) {
    ik_solve_fast<MAXD, M>(C, a.body, a.link, tpos, torn, lim != nullptr, lo, up, rg, rs, scr);
  } else {
    scr = rec + a.seed_floats;
    ik_solve(C, a.body, a.link, tpos, torn, a.use_orn, lim != nullptr, lo, up, rg, rs, scr);
  }
  for (int i = 0; i < ndb; i++) a.q_out[(size_t)e * ndb + i] = scr[i];
  if (!a.err) return;
  // the link frame in base coordinates at the returned q: walk up from the target link, composing parent <- child
  float R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, p[3] = {0, 0, 0};
  for (int gl = a.link; gl >= 0; gl = shc(C.link_i)[DG_LINK_I_W * gl + 1]) {
    const int dof = shc(C.link_i)[DG_LINK_I_W * gl + 3];
    float E[9], r[3], Et[9], Rn[9], t[3];
    joint_xform(C, gl, dof >= 0 ? scr[dof - d0] : 0.0f, E, r);
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) Et[3 * i + j] = E[3 * j + i];
    m_mul(Rn, Et, R); m_cpy(R, Rn); m_vec(t, Et, p); v_add(p, t, r);
  }
  const float* lfe = shc(C.link_f) + DG_LINK_F_W * a.link;
  float pos[3], dw[3], Rl[9], Rli[9], qi[4] = {-lfe[16], -lfe[17], -lfe[18], lfe[19]};
  m_vec(dw, R, lfe + 7); v_sub(pos, p, dw); q_to_mat(Rli, qi); m_mul(Rl, R, Rli);
  // the target in base coordinates, as the solve forms it
  const float *bp = ST(S_BPOS) + 3 * a.body, *bq = ST(S_BQUAT) + 4 * a.body;
  float Rb[9], d[3], tp[3], ep[3];
  q_to_mat(Rb, bq); v_sub(d, tpos, bp); mT_vec(tp, Rb, d); v_sub(ep, tp, pos);
  float ang = 0.f;
  if (a.use_orn) {
    float bqi[4] = {-bq[0], -bq[1], -bq[2], bq[3]}, tq[4], qc[4], qci[4], dq[4];
    q_mul(tq, bqi, torn); mat_to_q(qc, Rl); qci[0] = -qc[0]; qci[1] = -qc[1]; qci[2] = -qc[2]; qci[3] = qc[3];
    q_mul(dq, tq, qci);
    ang = 2 * atan2f(v_len(dq), fabsf(dq[3]));
  }
  a.err[2 * (size_t)e] = v_len(ep); a.err[2 * (size_t)e + 1] = ang;
}

}  // namespace dg
