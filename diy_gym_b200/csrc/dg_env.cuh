// dg_env.cuh - the per-environment step, written once for a TEAM of `nt` cooperating lanes.
//
// One environment is advanced by a team of nt lanes (nt = 1,2,4,...,32).  The code is a sequence of PHASES; inside
// a phase every lane works on its own items (bodies, M^-1 columns, shape pairs, constraint rows, add-on ops) and
// never reads what another lane writes in the same phase; between phases the lanes synchronise (a block barrier:
// see "the phase schedule" at the end of this file for how lanes map to threads).  The test-only CPU emulation
// (tests/emul) runs the same phases lane after lane, which is exactly the barrier semantics.
//
// What it computes replaces, for N environments at once, the reference's
//   DIYGym.step  (/root/reference/diy_gym/diy_gym.py:187-209):  add-on update -> p.stepSimulation() -> observe/reward/terminal
//   DIYGym.reset (/root/reference/diy_gym/diy_gym.py:130-148):  add-on reset -> hot-start steps -> observe
// with p.stepSimulation() configured as at diy_gym.py:76-82 (fixedTimeStep 1/240, numSubSteps 2, 150 solver sweeps).
// The physics is this repo's own fp32 engine (articulated-body forward dynamics, primitive contact generation,
// projected Gauss-Seidel on motor / limit / contact rows); its fp64 checker is oracle/bullet_restatement.c.
#pragma once
#include "dg_math.cuh"
#include "dg_scene.h"

namespace dg {

struct Env {
  const DevScene* sc;
  float* ws;          // team workspace, hot part (shared memory on the GPU)
  float* wg;          // team workspace, cold part (global memory, L1/L2 resident); regions with a negative offset live here
  float* st;          // this environment's state row  [S]
  float* pr;          // this environment's parameter row [P]
  const float* act;   // [n_act]
  float* obs;         // [n_obs]
  float* rew;         // [n_rew]
  uint8_t* term;      // [n_term]
  const int* link_i;  // link tables: the scene's global arrays, or the block's shared-memory copies on the GPU
  const float* link_f;
  const float* link_x;
  uint32_t seed;
  int env_id;
  bool active;        // false: no environment for this slot in this launch (barriers only)
  int grp0, grp1;     // environments of the block that share a warp in the row-space sweeps, as offsets (in workspaces) from this one: [grp0, grp1)
  unsigned long long opmask[2];   // bit k clear = action op k absent from this step's action dict (not updated)
  unsigned long long* dbg;        // phase timing (dg_debug_phase_cycles): [block][64] cycle sums keyed by source line & 63, or null
  unsigned* dropped;              // contacts lost to the max_contacts cap since the world was created (one counter per world), or null
  // split schedule (GPU only): the contact sweeps of this environment may be left to the sweep kernel (dg_solve_kernel)
  int split;                      // 1: environments whose rows fit a warp are deferred to the sweep kernel
  int* rs_lists; int rs_stride;   // deferred environments by sweep-kernel class: class c at rs_lists + c rs_stride (local indices), or null
  int* rs_count;                  // [RS_NCLS] their counts (atomically incremented)
  int e_local;                    // index of this environment in the launch
  unsigned* rs_used;              // counter of environment sub-steps solved in row space (any schedule), or null
  int no_hot;                     // reset launch without the hot-start steps (they follow as stage launches)
};

#define SC (*C.sc)
// Address-space hints: regions with a fixed home are addressed through pointers the compiler knows to be shared /
// global (LDS / LDG instead of generic loads); only the contact regions, whose home is chosen per scene, stay generic.
#if defined(__CUDA_ARCH__)
DG_HD float* as_shared(float* p) { __builtin_assume(__isShared(p)); return p; }
DG_HD float* as_global(float* p) { __builtin_assume(__isGlobal(p)); return p; }
template <class P> DG_HD const P* gc(const P* p) { __builtin_assume(__isGlobal(p)); return p; }
template <class P> DG_HD const P* shc(const P* p) { __builtin_assume(__isShared(p)); return p; }
#else
DG_HD float* as_shared(float* p) { return p; }
DG_HD float* as_global(float* p) { return p; }
template <class P> DG_HD const P* gc(const P* p) { return p; }
template <class P> DG_HD const P* shc(const P* p) { return p; }
#endif
#define WSH(C, off) (as_shared((C).ws) + (off))
#define WSG(C, off) (as_global((C).wg) + (off))
#define WSI(C) ((int*)as_shared((C).ws))
#define WSP(C, off) ((off) >= 0 ? (C).ws + (off) : (C).wg + ~(off))
#define WSIP(C, off) ((int*)WSP(C, off))
#define KIN(s) (WSG(C, SC.W_KIN) + 12 * (s))
#define LNK(gl) (WSG(C, SC.W_LINK) + LK_W * (gl))       // E9 r3 U6 D1 pad
#define ABA(s) (WSG(C, SC.X_ABA) + AB_W * (s))        // pA6 w3 v3 | A9 B9 C9 pad | acc6 pad2
#define LNX(gl) (WSG(C, SC.X_LNK) + LX_W * (gl))       // c6 u1 pad
#define DOF(k, d) (as_shared(C.ws)[SC.W_DOF + (k) * SC.nd + (d)])
#define BST(di) (WSH(C, SC.W_BST) + 13 * (di))
#define ST(name) (as_global(C.st) + DG_SO(C.sc, name))
#define PR(name) (as_global(C.pr) + DG_PO(C.sc, name))

DG_HD float clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }
DG_HD int float_as_int(float f) { union { float f; int i; } u; u.f = f; return u.i; }
DG_HD float int_as_float(int i) { union { float f; int i; } u; u.i = i; return u.f; }

// ------------------------------------------------------------------ load / store -------------------------------
// Copies the dynamic part of the state row into the workspace; static bodies that are not baked get their pose too.
DG_FN void phase_load(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  for (int i = ln; i < 13 * sc.ndyn; i += nt) {
    int di = i / 13, k = i - 13 * di, b = gc(sc.dyn_body)[di];
    float v;
    if (k < 3) v = ST(S_BPOS)[3 * b + k];
    else if (k < 7) v = ST(S_BQUAT)[4 * b + k - 3];
    else if (k < 10) v = ST(S_BVEL)[3 * b + k - 7];
    else v = ST(S_BOMEGA)[3 * b + k - 10];
    BST(di)[k] = v;
  }
  for (int d = ln; d < sc.nd; d += nt) {
    float qd = ST(S_QD)[d];
    DOF(D_Q, d) = ST(S_Q)[d]; DOF(D_QD, d) = qd; DOF(D_APPLIED, d) = ST(S_MAPPLIED)[d];
    DOF(D_TAU, d) = ST(S_JTORQUE)[d] - PR(P_JDAMP)[d] * qd;   // applied torque + joint damping, evaluated once per outer step
  }
  for (int f = ln; f < sc.nb; f += nt) {
    int s = gc(sc.frame_slot)[f];
    if (s < 0 || gc(sc.body_i)[DG_BODY_I_W * f] != 0) continue;
    float* K = KIN(s);                                        // static body with a per-environment pose
    q_to_mat(K, ST(S_BQUAT) + 4 * f); v_cpy(K + 9, ST(S_BPOS) + 3 * f);
  }
  if (ln == 0) for (int i = 0; i < WH_COUNT; i++) WSI(C)[sc.W_HDR + i] = 0;
}

// ------------------------------------------------------------------ kinematics ---------------------------------
// joint transform of link gl at coordinate q:  E = child_from_parent rotation, r = child COM in parent coordinates
DG_FN void joint_xform(const Env& C, int gl, float q, float* E, float* r) {
  const int* li = shc(C.link_i) + DG_LINK_I_W * gl; const float* lf = shc(C.link_f) + DG_LINK_F_W * gl; const float* R0 = shc(C.link_x) + 16 * gl;
  float Rrel[9], tmp[3];
  if (li[2] == 1) { float Ra[9]; axis_angle_mat(Ra, lf + 10, q, C.sc->precise != 0); m_mul(Rrel, R0, Ra); m_vec(tmp, Rrel, lf + 7); }
  else if (li[2] == 2) { m_cpy(Rrel, R0); float dd[3] = {lf[7] + lf[10] * q, lf[8] + lf[11] * q, lf[9] + lf[12] * q}; m_vec(tmp, R0, dd); }
  else { m_cpy(Rrel, R0); m_vec(tmp, R0, lf + 7); }
  v_add(r, lf + 4, tmp);
  E[0] = Rrel[0]; E[1] = Rrel[3]; E[2] = Rrel[6]; E[3] = Rrel[1]; E[4] = Rrel[4]; E[5] = Rrel[7]; E[6] = Rrel[2]; E[7] = Rrel[5]; E[8] = Rrel[8];
}
DG_HD int parent_slot(const int* li, int l0, int s0) { return li[1] < 0 ? s0 : s0 + 1 + (li[1] - l0); }

// ---- register-block loads / stores (128-bit when the address is 16-byte aligned, which every region base and
// every per-slot stride below guarantees) -------------------------------------------------------------------------
struct F4 { float x, y, z, w; };
DG_HD F4 ld4(const float* p) {
#if defined(__CUDA_ARCH__)
  float4 v = *reinterpret_cast<const float4*>(p); F4 o = {v.x, v.y, v.z, v.w}; return o;
#else
  F4 o = {p[0], p[1], p[2], p[3]}; return o;
#endif
}
DG_HD void st4(float* p, float x, float y, float z, float w) {
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<float4*>(p) = make_float4(x, y, z, w);
#else
  p[0] = x; p[1] = y; p[2] = z; p[3] = w;
#endif
}
template <int N> DG_HD void ldn(const float* p, float* o) {   // N multiple of 4
#pragma unroll
  for (int c = 0; c < N / 4; c++) { F4 v = ld4(p + 4 * c); o[4 * c] = v.x; o[4 * c + 1] = v.y; o[4 * c + 2] = v.z; o[4 * c + 3] = v.w; }
}
template <int N> DG_HD void stn(float* p, const float* v) {
#pragma unroll
  for (int c = 0; c < N / 4; c++) st4(p + 4 * c, v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}

// world pose and body-frame spatial velocity of every frame of dynamic body b; with BIAS also the first ABA pass
// (bias forces, rigid-body inertias, velocity-product accelerations), fused so that nothing is re-read
template <bool BIAS>
DG_FN void fk_vel_body(const Env& C, int b) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
  const int kind = bi[0], l0 = bi[1], nlb = bi[2], s0 = bp[BP_SLOT];
  const float* bs = BST(bp[BP_DI]);
  const float *mass = PR(P_MASS), *inertia = PR(P_INERTIA);
  const float kl = PR(P_LINDAMP)[b], ka = PR(P_ANGDAMP)[b];
  float Kp[12], Vp[6];      // pose (R 9, p 3) and velocity (w 3, v 3) of the previously visited frame
  q_to_mat(Kp, bs + 3); v_cpy(Kp + 9, bs);
  mT_vec(Vp, Kp, bs + 10); mT_vec(Vp + 3, Kp, bs + 7);
  int prev = s0;
  for (int k = -1; k < nlb; k++) {
    const int s = s0 + 1 + k, f = k < 0 ? b : sc.nb + l0 + k;
    float K[12], V[6], cacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (k < 0) {
      for (int i = 0; i < 12; i++) K[i] = Kp[i];
      for (int i = 0; i < 6; i++) V[i] = Vp[i];
    } else {
      const int gl = l0 + k; const int* li = shc(C.link_i) + DG_LINK_I_W * gl; const float* lx = shc(C.link_x) + 16 * gl;
      const int ps = parent_slot(li, l0, s0), dof = li[3];
      if (ps != prev) { ldn<12>(KIN(ps), Kp); const float* pv = ABA(ps) + AB_WV; for (int i = 0; i < 6; i++) Vp[i] = pv[i]; }
      float E[9], r[3], t[3], t2[3];
      joint_xform(C, gl, dof >= 0 ? DOF(D_Q, dof) : 0.f, E, r);
      float* L = LNK(gl);
      st4(L, E[0], E[1], E[2], E[3]); st4(L + 4, E[4], E[5], E[6], E[7]); st4(L + 8, E[8], r[0], r[1], r[2]);
      m_mulT(K, Kp, E);
      m_vec(t, Kp, r); v_add(K + 9, Kp + 9, t);
      m_vec(V, E, Vp);
      v_cross(t, Vp, r); v_add(t2, Vp + 3, t); m_vec(V + 3, E, t2);
      if (dof >= 0) {
        const float qd = DOF(D_QD, dof);
        if (BIAS) { float sa[3], sl[3]; v_scale(sa, lx + 9, qd); v_scale(sl, lx + 12, qd); v_cross(cacc, V, sa); v_cross(cacc + 3, V, sl); v_cross(t2, V + 3, sa); v_add(cacc + 3, cacc + 3, t2); }
        v_madd(V, lx + 9, qd); v_madd(V + 3, lx + 12, qd);
      }
      if (BIAS) stn<8>(LNX(gl), cacc);
    }
    stn<12>(KIN(s), K);
    float* X = ABA(s);
    if (!BIAS) {
      for (int i = 0; i < 6; i++) X[AB_WV + i] = V[i];
    } else if (k < 0 && kind != 2) {
      float z[40]; for (int i = 0; i < 40; i++) z[i] = 0.f;
      for (int i = 0; i < 6; i++) z[AB_WV + i] = V[i];
      stn<40>(X, z);
    } else {
      // SEM_WRENCH_FIRST_SUBSTEP: applied wrenches act during the first internal sub-step only
      const float wsc = ((sc.sem & SEM_WRENCH_FIRST_SUBSTEP) && WSI(C)[sc.W_HDR + WH_SUB] > 0) ? 0.f : 1.f;
      const float efv[3] = {wsc * ST(S_EXTF)[3 * f], wsc * ST(S_EXTF)[3 * f + 1], wsc * ST(S_EXTF)[3 * f + 2]}, etv[3] = {wsc * ST(S_EXTT)[3 * f], wsc * ST(S_EXTT)[3 * f + 1], wsc * ST(S_EXTT)[3 * f + 2]};
      const float *ef = efv, *et = etv;
      const float m = mass[f]; const float* I = inertia + 3 * f; const float *w = V, *v = V + 3;
      float Iw[3] = {I[0] * w[0], I[1] * w[1], I[2] * w[2]}, t[3], fw[3], pa[3], pl[3];
      v_cross(pa, w, Iw);
      v_cross(t, w, v); v_scale(pl, t, m);
      fw[0] = sc.g[0] * m + ef[0]; fw[1] = sc.g[1] * m + ef[1]; fw[2] = sc.g[2] * m + ef[2];
      mT_vec(t, K, fw); v_sub(pl, pl, t);
      mT_vec(t, K, et); v_sub(pa, pa, t);
      const float wn = v_len(w), vn = v_len(v);
      const bool dlin = (sc.sem & SEM_DAMPING_LINEAR) != 0;   // damping -m v k instead of -m v (k + k |v|)
      v_madd(pa, Iw, dlin ? ka : ka + ka * wn);
      float mv[3]; v_scale(mv, v, m); v_madd(pl, mv, dlin ? kl : kl + kl * vn);
      float z[40]; for (int i = 0; i < 40; i++) z[i] = 0.f;
      for (int i = 0; i < 3; i++) { z[AB_PA + i] = pa[i]; z[AB_PA + 3 + i] = pl[i]; z[AB_WV + i] = w[i]; z[AB_WV + 3 + i] = v[i]; }
      z[AB_A] = I[0]; z[AB_A + 4] = I[1]; z[AB_A + 8] = I[2]; z[AB_C] = m; z[AB_C + 4] = m; z[AB_C + 8] = m;
      stn<40>(X, z);
    }
    for (int i = 0; i < 12; i++) Kp[i] = K[i];
    for (int i = 0; i < 6; i++) Vp[i] = V[i];
    prev = s;
  }
}

// ------------------------------------------------------------------ articulated-body algorithm -----------------
DG_HD void ia_mul(const float* A, const float* B, const float* Cm, const float* a, const float* l, float* n, float* f) {
  float t[3]; m_vec(n, A, a); m_vec(t, B, l); v_add(n, n, t); mT_vec(f, B, a); m_vec(t, Cm, l); v_add(f, f, t);
}
// Gauss-Jordan inverse with partial pivoting of the n x n matrix M (destroyed); both live in the workspace
DG_FN int invert_small(float* M, int n, float* inv) {
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) inv[i * n + j] = (i == j) ? 1.f : 0.f;
  for (int c = 0; c < n; c++) {
    int p = c;
    for (int r2 = c + 1; r2 < n; r2++) if (fabsf(M[r2 * n + c]) > fabsf(M[p * n + c])) p = r2;
    if (fabsf(M[p * n + c]) < 1e-30f) return -1;
    if (p != c) for (int j = 0; j < n; j++) { float t = M[c * n + j]; M[c * n + j] = M[p * n + j]; M[p * n + j] = t; t = inv[c * n + j]; inv[c * n + j] = inv[p * n + j]; inv[p * n + j] = t; }
    float d = 1.0f / M[c * n + c];
    for (int j = 0; j < n; j++) { M[c * n + j] *= d; inv[c * n + j] *= d; }
    for (int r2 = 0; r2 < n; r2++) if (r2 != c) {
      float fct = M[r2 * n + c];
      if (fct != 0.f) for (int j = 0; j < n; j++) { M[r2 * n + j] -= fct * M[c * n + j]; inv[r2 * n + j] -= fct * inv[c * n + j]; }
    }
  }
  return 0;
}

// inverse of a symmetric positive definite N x N matrix held in registers: A = L L^T, L^-1 by forward substitution,
// A^-1 = L^-T L^-1.  Every index is a compile-time constant after unrolling.  (A pivot that is not positive - a body without
// mass - is clamped: the result is then meaningless but finite, as with the pivoting elimination it replaces.)
template <int N> DG_HD void inv_spd(const float (&A)[N][N], float (&Out)[N][N]) {
  float L[N][N], Li[N][N], invd[N];
#pragma unroll
  for (int j = 0; j < N; j++) {
    float d = A[j][j];
#pragma unroll
    for (int k = 0; k < N; k++) if (k < j) d -= L[j][k] * L[j][k];
    const float ljj = sqrtf(fmaxf(d, 1e-30f)), inv = 1.0f / ljj;
    L[j][j] = ljj; invd[j] = inv;
#pragma unroll
    for (int i = 0; i < N; i++) if (i > j) {
      float v = A[i][j];
#pragma unroll
      for (int k = 0; k < N; k++) if (k < j) v -= L[i][k] * L[j][k];
      L[i][j] = v * inv;
    }
  }
#pragma unroll
  for (int j = 0; j < N; j++) {
    Li[j][j] = invd[j];
#pragma unroll
    for (int i = 0; i < N; i++) if (i > j) {
      float v = 0.f;
#pragma unroll
      for (int k = 0; k < N; k++) if (k >= j && k < i) v -= L[i][k] * Li[k][j];
      Li[i][j] = v * invd[i];
    }
  }
#pragma unroll
  for (int i = 0; i < N; i++)
#pragma unroll
    for (int j = 0; j < N; j++) {
      float v = 0.f;
#pragma unroll
      for (int k = 0; k < N; k++) if (k >= i && k >= j) v += Li[k][i] * Li[k][j];
      Out[i][j] = v;
    }
}
// forward dynamics of dynamic body b (passes 2 and 3 of the ABA; pass 1 ran inside fk_vel_body<true>), then the
// velocity half of the semi-implicit Euler step.  Every per-link record is pulled into registers with 128-bit loads,
// worked on there, and written back once.
DG_FN void aba_body(const Env& C, int b, float h) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
  const int kind = bi[0], l0 = bi[1], nlb = bi[2], s0 = bp[BP_SLOT], di = bp[BP_DI];
  // pass 2: articulated inertias, leaves to root
  for (int k = nlb - 1; k >= 0; k--) {
    const int gl = l0 + k, s = s0 + 1 + k; const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
    const int ps = parent_slot(li, l0, s0);
    float Xr[40], Lr[12], cx[8];
    ldn<40>(ABA(s), Xr); ldn<12>(LNK(gl), Lr); ldn<8>(LNX(gl), cx);
    float* Aa = Xr + AB_A; float* Ba = Xr + AB_B; float* Ca = Xr + AB_C; const float* pA = Xr + AB_PA;
    float pa[6], n[3], fo[3];
    if (li[3] >= 0) {
      const float* lx = shc(C.link_x) + 16 * gl; const float *sa = lx + 9, *sl = lx + 12;
      float U[6];
      ia_mul(Aa, Ba, Ca, sa, sl, U, U + 3);
      const float D = v_dot(sa, U) + v_dot(sl, U + 3);
      const float uu = DOF(D_TAU, li[3]) - (v_dot(sa, pA) + v_dot(sl, pA + 3));
      float* L = LNK(gl);
      st4(L + 12, U[0], U[1], U[2], U[3]); st4(L + 16, U[4], U[5], D, 0.f);
      LNX(gl)[6] = uu;
      const float Dinv = 1.0f / D;
#pragma unroll
      for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) { Aa[3 * i + j] -= U[i] * U[j] * Dinv; Ba[3 * i + j] -= U[i] * U[3 + j] * Dinv; Ca[3 * i + j] -= U[3 + i] * U[3 + j] * Dinv; }
      ia_mul(Aa, Ba, Ca, cx, cx + 3, n, fo);
      for (int i = 0; i < 3; i++) { pa[i] = pA[i] + n[i] + U[i] * uu * Dinv; pa[3 + i] = pA[3 + i] + fo[i] + U[3 + i] * uu * Dinv; }
    } else {
      ia_mul(Aa, Ba, Ca, cx, cx + 3, n, fo);
      for (int i = 0; i < 3; i++) { pa[i] = pA[i] + n[i]; pa[3 + i] = pA[3 + i] + fo[i]; }
    }
    // transform to the parent: rotate the blocks by E^T (.) E, then shift by r
    const float* E = Lr; const float* r = Lr + 9;
    float T1[9], Ar[9], Br[9], Cr[9];
    mT_mul(T1, E, Aa); m_mul(Ar, T1, E); mT_mul(T1, E, Ba); m_mul(Br, T1, E); mT_mul(T1, E, Ca); m_mul(Cr, T1, E);
    const float Kx[9] = {0, -r[2], r[1], r[2], 0, -r[0], -r[1], r[0], 0};
    float KC[9], BK[9], KBt[9], KCK[9];
    m_mul(KC, Kx, Cr); m_mul(BK, Br, Kx); m_mulT(KBt, Kx, Br); m_mul(KCK, KC, Kx);
    float fp[3], np_[3], t[3];
    mT_vec(fp, E, pa + 3); mT_vec(np_, E, pa); v_cross(t, r, fp); v_add(np_, np_, t);
    float* P = ABA(ps);
    float Pr[40];
    ldn<40>(P, Pr);
    for (int i = 0; i < 9; i++) { Pr[AB_A + i] += Ar[i] - BK[i] + KBt[i] - KCK[i]; Pr[AB_B + i] += Br[i] + KC[i]; Pr[AB_C + i] += Cr[i]; }
    for (int i = 0; i < 3; i++) { Pr[AB_PA + i] += np_[i]; Pr[AB_PA + 3 + i] += fp[i]; }
    stn<40>(P, Pr);
  }
  // base acceleration
  float* X0 = ABA(s0); float* a0 = X0 + AB_ACC;
#if defined(DG_OLD_INV)
  if (kind == 2) {
    float* M = WSG(C, sc.X_I0T) + bp[BP_I0OFF]; float* Iv = WSG(C, sc.W_I0) + bp[BP_I0OFF];
    const float *A = X0 + AB_A, *B = X0 + AB_B, *Cm = X0 + AB_C;
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { M[6 * i + j] = A[3 * i + j]; M[6 * i + 3 + j] = B[3 * i + j]; M[6 * (3 + i) + j] = B[3 * j + i]; M[6 * (3 + i) + 3 + j] = Cm[3 * i + j]; }
    invert_small(M, 6, Iv);
    for (int i = 0; i < 6; i++) { float sum = 0.f; for (int j = 0; j < 6; j++) sum -= Iv[6 * i + j] * X0[AB_PA + j]; a0[i] = sum; }
  } else for (int i = 0; i < 6; i++) a0[i] = 0.f;
#else
  if (kind == 2) {
    // inverse of the base's articulated inertia [A B; B^T C] (symmetric positive definite): Cholesky in registers, fully
    // unrolled (round 1 ran a pivoting Gauss-Jordan on the cold workspace: ~300 dependent memory operations per body)
    float* Iv = WSG(C, sc.W_I0) + bp[BP_I0OFF];
    float Xr[40]; ldn<40>(X0, Xr);
    const float *A = Xr + AB_A, *B = Xr + AB_B, *Cm = Xr + AB_C;
    float M[6][6], Inv[6][6];
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
      for (int j = 0; j < 3; j++) { M[i][j] = A[3 * i + j]; M[i][3 + j] = B[3 * i + j]; M[3 + i][j] = B[3 * j + i]; M[3 + i][3 + j] = Cm[3 * i + j]; }
    inv_spd<6>(M, Inv);
    float iv[36];
#pragma unroll
    for (int i = 0; i < 6; i++)
#pragma unroll
      for (int j = 0; j < 6; j++) iv[6 * i + j] = Inv[i][j];
    stn<36>(Iv, iv);
#pragma unroll
    for (int i = 0; i < 6; i++) { float sum = 0.f;
#pragma unroll
      for (int j = 0; j < 6; j++) sum -= Inv[i][j] * Xr[AB_PA + j];
      a0[i] = sum; }
  } else for (int i = 0; i < 6; i++) a0[i] = 0.f;
#endif
  // pass 3: accelerations, root to leaves
  float ap[8]; int prev = s0;
  ldn<8>(a0, ap);
  for (int k = 0; k < nlb; k++) {
    const int gl = l0 + k, s = s0 + 1 + k; const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
    const int ps = parent_slot(li, l0, s0);
    if (ps != prev) ldn<8>(ABA(ps) + AB_ACC, ap);
    float Lr[20], cx[8];
    ldn<20>(LNK(gl), Lr); ldn<8>(LNX(gl), cx);
    float t[3], t2[3], acc[8];
    m_vec(acc, Lr, ap); v_cross(t, ap, Lr + 9); v_add(t2, ap + 3, t); m_vec(acc + 3, Lr, t2);
    v_add(acc, acc, cx); v_add(acc + 3, acc + 3, cx + 3);
    if (li[3] >= 0) {
      const float* lx = shc(C.link_x) + 16 * gl;
      const float qdd = (cx[6] - (v_dot(Lr + 12, acc) + v_dot(Lr + 15, acc + 3))) / Lr[18];
      DOF(D_QD, li[3]) += h * qdd;            // velocity half of the semi-implicit Euler step
      v_madd(acc, lx + 9, qdd); v_madd(acc + 3, lx + 12, qdd);
    }
    acc[6] = 0.f; acc[7] = 0.f;
    stn<8>(ABA(s) + AB_ACC, acc);
    for (int i = 0; i < 8; i++) ap[i] = acc[i];
    prev = s;
  }
  // velocity update of a floating base
  if (kind == 2) {
    const float* K0 = KIN(s0); float* bs = BST(di); float t[3], lin[3], aw[3];
    v_cross(t, X0 + AB_WV, X0 + AB_WV + 3); v_add(lin, a0 + 3, t);
    m_vec(aw, K0, a0); v_madd(bs + 10, aw, h);
    m_vec(aw, K0, lin); v_madd(bs + 7, aw, h);
  }
}

// joint reaction wrench of every link of body b: f = I^A a + p^A in the link's COM frame, [force(3), torque(3)], from the
// forward-dynamics pass that just ran (what p.getJointState(...)[2] reports, force_torque_sensor.py:21-23)
DG_FN void joint_reactions(const Env& C, int b) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int l0 = bi[1], nlb = bi[2], s0 = gc(sc.body_plan)[BP_W * b + BP_SLOT];
  for (int k = 0; k < nlb; k++) {
    float X[48], n[3], f[3];
    ldn<48>(ABA(s0 + 1 + k), X);
    ia_mul(X + AB_A, X + AB_B, X + AB_C, X + AB_ACC, X + AB_ACC + 3, n, f);
    float* o = ST(S_JREACT) + 6 * (l0 + k);
    for (int i = 0; i < 3; i++) { o[i] = X[AB_PA + 3 + i] + f[i]; o[3 + i] = X[AB_PA + i] + n[i]; }
  }
}
DG_FN void phase_dynamics(const Env& C, int ln, int nt, float h) {
  for (int di = ln; di < SC.ndyn; di += nt) { int b = gc(SC.dyn_body)[di]; fk_vel_body<true>(C, b); aba_body(C, b, h); if (SC.need_react) joint_reactions(C, b); }
}

// One column of M^-1 of body b: response of the generalized velocity to a unit generalized impulse at coordinate col.
// Coordinates: floating bodies [torque_world(3), force_world(3), joints...], fixed-base bodies [joints...].
DG_FN void minv_column(const Env& C, int b, int col, float* scr) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
  const int kind = bi[0], l0 = bi[1], nlb = bi[2], d0 = bi[3], s0 = bp[BP_SLOT], g = bp[BP_GDIM], gs = bp[BP_GS];
  const int jo = kind == 2 ? 6 : 0;
  float* out = WSH(C, sc.W_MINV) + bp[BP_MINVOFF] + col * gs;
  for (int i = g; i < gs; i++) out[i] = 0.f;
  // u of every link and the stack of parent accelerations (indexed by depth + 1, 0 = base) live in THREAD-LOCAL memory: the pass
  // down reads what it stored a few instructions earlier, and a global store -> load round trip through L2 at every branch of the
  // tree was the longest stall of this phase (local memory stays in L1).  Caps checked by HostScene::build.
  (void)scr;
  float uu[DG_MINV_MAXL], ast[6 * DG_MINV_MAXD];
  for (int k = 0; k < nlb; k++) uu[k] = 0.f;
  float p[6] = {0, 0, 0, 0, 0, 0};
  if (col >= jo) {
    int k0 = -1;
    for (int k = 0; k < nlb; k++) if (shc(C.link_i)[DG_LINK_I_W * (l0 + k) + 3] == d0 + col - jo) { k0 = k; break; }
    for (int k = k0; k >= 0;) {
      const int gl = l0 + k; const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
      float L[20]; ldn<20>(LNK(gl), L);
      float pa[6] = {p[0], p[1], p[2], p[3], p[4], p[5]};
      if (li[3] >= 0) {
        const float* lx = shc(C.link_x) + 16 * gl;
        const float u1 = (k == k0 ? 1.f : 0.f) - (v_dot(lx + 9, pa) + v_dot(lx + 12, pa + 3));
        uu[k] = u1; const float s = u1 / L[18];
        for (int i = 0; i < 6; i++) pa[i] += L[12 + i] * s;
      }
      float fp[3], np_[3], t[3];
      mT_vec(fp, L, pa + 3); mT_vec(np_, L, pa); v_cross(t, L + 9, fp); v_add(np_, np_, t);
      v_cpy(p, np_); v_cpy(p + 3, fp);
      k = li[1] < 0 ? -1 : li[1] - l0;
    }
  }
  float a0[6];
  if (kind == 2) {
    float K0[12]; ldn<12>(KIN(s0), K0); const float* Iv = WSG(C, sc.W_I0) + bp[BP_I0OFF];
    float gen[6] = {0, 0, 0, 0, 0, 0}, rhs[6], t[3];
    for (int i = 0; i < 6; i++) gen[i] = (i == col) ? 1.f : 0.f;
    mT_vec(t, K0, gen); v_sub(rhs, t, p); mT_vec(t, K0, gen + 3); v_sub(rhs + 3, t, p + 3);
    for (int i = 0; i < 6; i++) { float s = 0.f; for (int j = 0; j < 6; j++) s += Iv[6 * i + j] * rhs[j]; a0[i] = s; }
    m_vec(out, K0, a0); m_vec(out + 3, K0, a0 + 3);
  } else for (int i = 0; i < 6; i++) a0[i] = 0.f;
  for (int i = 0; i < 6; i++) ast[i] = a0[i];
  float ap[6] = {a0[0], a0[1], a0[2], a0[3], a0[4], a0[5]}; int prev_dep = -1;   // registers hold a of depth prev_dep
  for (int k = 0; k < nlb; k++) {
    const int gl = l0 + k; const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
    const int dep = gc(sc.link_depth)[gl];
    if (dep - 1 != prev_dep) { const float* src = ast + 6 * dep; for (int i = 0; i < 6; i++) ap[i] = src[i]; }
    float L[20]; ldn<20>(LNK(gl), L);
    float t[3], t2[3], aa[3], al[3];
    m_vec(aa, L, ap); v_cross(t, ap, L + 9); v_add(t2, ap + 3, t); m_vec(al, L, t2);
    if (li[3] >= 0) {
      const float* lx = shc(C.link_x) + 16 * gl;
      const float qdd = (uu[k] - (v_dot(L + 12, aa) + v_dot(L + 15, al))) / L[18];
      out[jo + li[3] - d0] = qdd;
      v_madd(aa, lx + 9, qdd); v_madd(al, lx + 12, qdd);
    }
    float* ak = ast + 6 * (dep + 1);
    v_cpy(ak, aa); v_cpy(ak + 3, al);
    v_cpy(ap, aa); v_cpy(ap + 3, al); prev_dep = dep;
  }
}
DG_FN void phase_minv(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  float* scr = WSG(C, sc.X_MSCR) + sc.mscr_stride * ln;
  int item = 0;
  for (int di = 0; di < sc.ndyn; di++) {
    int b = gc(sc.dyn_body)[di], g = gc(sc.body_plan)[BP_W * b + BP_GDIM];
    for (int col = 0; col < g; col++, item++) if (item % nt == ln) minv_column(C, b, col, scr);
  }
}

// ------------------------------------------------------------------ collision ----------------------------------
struct Ct { int fa, fb; float pa[3], pb[3], n[3], dist, mu; };

DG_FN void shape_pose(const Env& C, int s, const float** R, const float** p) {
  int sl = gc(SC.shape_slot)[s];
  const float* w = sl >= 0 ? WSP(C, SC.X_SHW) + 12 * sl : gc(SC.shape_wb) + 12 * s;
  *R = w; *p = w + 9;
}
DG_FN void phase_shape_world(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  for (int s = ln; s < sc.ns; s += nt) {
    int sl = gc(sc.shape_slot)[s];
    if (sl < 0) continue;
    const float* sf = gc(sc.shape_f) + DG_SHAPE_F_W * s; const float* K = KIN(gc(sc.frame_slot)[gc(sc.shape_i)[DG_SHAPE_I_W * s + 1]]);
    float* w = WSP(C, sc.X_SHW) + 12 * sl; float Rl[9], R[9], t[3];
    q_to_mat(Rl, sf + 3); m_mul(R, K, Rl); m_cpy(w, R); m_vec(t, K, sf); v_add(w + 9, K + 9, t);
  }
  int nw = (sc.npair + 31) / 32;
  for (int i = ln; i < nw; i += nt) WSIP(C, sc.X_SURV)[i] = 0;
  if (ln == 0) { int* hdr = WSI(C) + sc.W_HDR; hdr[WH_NCONTACT] = 0; hdr[WH_RS_R] = 0; hdr[WH_RS_DEFER] = 0; }
}
DG_HD void ct_add(Ct* list, int* n, int cap, int fa, int fb, const float* pa, const float* pb, const float* nrm, float dist, float mu, float margin) {
  if (dist > margin || *n >= cap) return;
  Ct* c = &list[(*n)++]; c->fa = fa; c->fb = fb; v_cpy(c->pa, pa); v_cpy(c->pb, pb); v_cpy(c->n, nrm); c->dist = dist; c->mu = mu;
}
DG_FN int sphere_box(const float* c, float r, const float* Rb, const float* pb, const float* h, float* pa_out, float* pb_out, float* n, float* dist) {
  float d[3], cl[3], q[3]; v_sub(d, c, pb); mT_vec(cl, Rb, d);
  int inside = 1;
  for (int i = 0; i < 3; i++) { q[i] = cl[i]; if (q[i] > h[i]) { q[i] = h[i]; inside = 0; } else if (q[i] < -h[i]) { q[i] = -h[i]; inside = 0; } }
  float nl[3] = {0, 0, 0};
  if (!inside) {
    float dv[3]; v_sub(dv, cl, q); float len = v_len(dv);
    if (len < 1e-12f) return 0;
    v_scale(nl, dv, 1.0f / len); *dist = len - r;
  } else {
    int ax = 0; float best = 1e30f;
    for (int i = 0; i < 3; i++) { float pen = h[i] - fabsf(cl[i]); if (pen < best) { best = pen; ax = i; } }
    float sg = cl[ax] >= 0 ? 1.0f : -1.0f;
    for (int i = 0; i < 3; i++) if (i == ax) { nl[i] = sg; q[i] = sg * h[i]; }
    *dist = -best - r;
  }
  m_vec(n, Rb, nl); float t[3]; m_vec(t, Rb, q); v_add(pb_out, pb, t);
  v_scale(t, n, -r); v_add(pa_out, c, t);
  return 1;
}
DG_FN int point_box(const float* p, const float* Rb, const float* pb, const float* h, float margin, float* pb_out, float* n, float* dist) {
  float d[3], pl[3]; v_sub(d, p, pb); mT_vec(pl, Rb, d);
  int ax = 0; float best = 1e30f;
  for (int i = 0; i < 3; i++) { float pen = h[i] - fabsf(pl[i]); if (pen < -margin) return 0; if (pen < best) { best = pen; ax = i; } }
  float nl[3] = {0, 0, 0}, q[3] = {pl[0], pl[1], pl[2]};
  float sg = pl[ax] >= 0 ? 1.0f : -1.0f;
  for (int i = 0; i < 3; i++) if (i == ax) { nl[i] = sg; q[i] = sg * h[i]; }
  m_vec(n, Rb, nl); float t[3]; m_vec(t, Rb, q); v_add(pb_out, pb, t); *dist = -best;
  return 1;
}
DG_FN void seg_closest(const float* p1, const float* d1, const float* p2, const float* d2, float* s, float* t) {
  float r[3]; v_sub(r, p1, p2);
  float a = v_dot(d1, d1), e = v_dot(d2, d2), f = v_dot(d2, r);
  if (a <= 1e-18f && e <= 1e-18f) { *s = *t = 0; return; }
  if (a <= 1e-18f) { *s = 0; *t = clampf(f / e, 0.f, 1.f); return; }
  float c = v_dot(d1, r);
  if (e <= 1e-18f) { *t = 0; *s = clampf(-c / a, 0.f, 1.f); return; }
  float b = v_dot(d1, d2), den = a * e - b * b;
  *s = den > 1e-18f ? clampf((b * f - c * e) / den, 0.f, 1.f) : 0.0f;
  *t = (b * (*s) + f) / e;
  if (*t < 0) { *t = 0; *s = clampf(-c / a, 0.f, 1.f); } else if (*t > 1) { *t = 1; *s = clampf((b - c) / a, 0.f, 1.f); }
}
DG_FN void as_capsule(int type, const float* dims, const float* R, const float* p, float* e0, float* e1, float* rad) {
  float half = 0; *rad = dims[0];
  if (type == SHAPE_CAPSULE) half = dims[1];
  else if (type == SHAPE_CYLINDER) half = dims[1] - dims[0] > 0 ? dims[1] - dims[0] : 0;
  float ax[3] = {R[2] * half, R[5] * half, R[8] * half};
  v_sub(e0, p, ax); v_add(e1, p, ax);
}
DG_HD bool pair_in_reach(const Env& C, int sa, int sb) {
  const float *Ra, *pa, *Rb, *pb;
  shape_pose(C, sa, &Ra, &pa); shape_pose(C, sb, &Rb, &pb);
  float dc[3]; v_sub(dc, pa, pb);
  const float ra = gc(SC.shape_f)[DG_SHAPE_F_W * sa + 11], rb = gc(SC.shape_f)[DG_SHAPE_F_W * sb + 11];
  float reach = ra + rb + SC.margin;
  if (v_dot(dc, dc) > reach * reach) return false;
  // a true box (no hull) is tested itself, not its bounding ball: the other shape lies inside the ball of its radius about its
  // origin, so nothing of the pair can be within the margin unless that origin is within radius + margin of the box (a large
  // table under a robot arm otherwise lets every link of the arm through to the narrow phase)
  for (int side = 0; side < 2; side++) {
    const int sx = side ? sa : sb;   // the box
    const int* ix = gc(SC.shape_i) + DG_SHAPE_I_W * sx;
    if (ix[2] != SHAPE_BOX || ix[5] > 0) continue;
    const float *Rx = side ? Ra : Rb, *px = side ? pa : pb, *po = side ? pb : pa; const float* h = gc(SC.shape_f) + DG_SHAPE_F_W * sx + 7;
    float d[3], pl[3]; v_sub(d, po, px); mT_vec(pl, Rx, d);
    float d2 = 0.f;
    for (int i = 0; i < 3; i++) { const float ex = fabsf(pl[i]) - h[i]; if (ex > 0.f) d2 += ex * ex; }
    const float r = (side ? rb : ra) + SC.margin;
    if (d2 > r * r) return false;
  }
  return true;
}
// ---- reduced convex hulls (mesh links; model.py:65 loads them as btConvexHullShape) ----------------------------------------
// signed distance of world point p to the hull (R, pos; planes n . x <= d in its own frame): the largest plane distance.  Inside or
// within `margin`: returns 1 with the outward normal of that plane (world), the point moved onto it, and the (negative) distance.
DG_FN int point_hull(const float* p, const float* R, const float* pos, const float* planes, int np_, float margin, float* surf, float* n, float* dist) {
  float d[3], pl[3]; v_sub(d, p, pos); mT_vec(pl, R, d);
  float best = -1e30f; int bi = 0;
  // (a point beyond the margin of ANY plane is outside: leave at the first such plane - most vertices of a pair in reach are)
  for (int k = 0; k < np_; k++) { const float* q = planes + 4 * k; const float s = q[0] * pl[0] + q[1] * pl[1] + q[2] * pl[2] - q[3]; if (s > margin) return 0; if (s > best) { best = s; bi = k; } }
  m_vec(n, R, planes + 4 * bi); *dist = best;
  surf[0] = p[0] - n[0] * best; surf[1] = p[1] - n[1] * best; surf[2] = p[2] - n[2] * best;
  return 1;
}
// Convex pair with at least one hull (the other a hull or a box): the vertices of each that lie inside the other (edge-edge
// contacts are not generated, as in the box-box routine below); candidates in `loc`, the caller keeps the deepest four.
// Contact convention: (pa on A, pb on B, normal from B towards A).
DG_FN void collide_convex(const Env& C, const int* ia, const float* fa, const float* Ra, const float* pa, const int* ib, const float* fb, const float* Rb, const float* pb,
                          float mu, float margin, Ct* loc, int* nloc) {
  const float* H = gc(SC.hull_f);
  for (int side = 0; side < 2; side++) {
    // X: the shape whose vertices are tested, Y: the shape they are tested against
    const int* ix = side ? ib : ia; const int* iy = side ? ia : ib; const float* fx = side ? fb : fa; const float* fy = side ? fa : fb;
    const float *Rx = side ? Rb : Ra, *px = side ? pb : pa, *Ry = side ? Ra : Rb, *py = side ? pa : pb;
    const int nvx = ix[5] > 0 ? ix[5] : 8;
    const float reach2 = (fy[11] + margin) * (fy[11] + margin);   // Y lies inside the ball of radius fy[11] about its origin (compiler/scene.py)
    for (int k = 0; k < nvx; k++) {
      float vl[3], t[3], pt[3], surf[3], n[3], dist;
      if (ix[5] > 0) { const float* v = H + ix[4] + 3 * k; vl[0] = v[0]; vl[1] = v[1]; vl[2] = v[2]; }
      else { vl[0] = (k & 1 ? 1 : -1) * fx[7]; vl[1] = (k & 2 ? 1 : -1) * fx[8]; vl[2] = (k & 4 ? 1 : -1) * fx[9]; }
      m_vec(t, Rx, vl); v_add(pt, px, t);
      { float dy[3]; v_sub(dy, pt, py); if (v_dot(dy, dy) > reach2) continue; }   // a vertex farther than that cannot be within the margin of Y
      const int hit = iy[5] > 0 ? point_hull(pt, Ry, py, H + iy[6], iy[7], margin, surf, n, &dist) : point_box(pt, Ry, py, fy + 7, margin, surf, n, &dist);
      if (!hit) continue;
      if (side == 0) ct_add(loc, nloc, 16, ia[1], ib[1], pt, surf, n, dist, mu, margin);                       // vertex of A in B: normal of B
      else { float nn[3]; v_scale(nn, n, -1.0f); ct_add(loc, nloc, 16, ia[1], ib[1], surf, pt, nn, dist, mu, margin); }   // vertex of B in A
    }
  }
}
// narrow phase of one shape pair; writes at most 4 contacts into out, returns the count
DG_FN int collide_pair(const Env& C, int sa, int sb, Ct* out) {
  const DevScene& sc = SC;
  const int *ia = gc(sc.shape_i) + DG_SHAPE_I_W * sa, *ib = gc(sc.shape_i) + DG_SHAPE_I_W * sb;
  const float *fa = gc(sc.shape_f) + DG_SHAPE_F_W * sa, *fb = gc(sc.shape_f) + DG_SHAPE_F_W * sb;
  const float *Ra, *pa, *Rb, *pb;
  shape_pose(C, sa, &Ra, &pa); shape_pose(C, sb, &Rb, &pb);
  float margin = sc.margin;
  int ta = ia[2], tb = ib[2];
  float mu = PR(P_FRICTION)[sa] * PR(P_FRICTION)[sb];
  int nt_ = 0;
  float ca[3], cb[3], n[3], dist;
  // mesh links: reduced hull against a box or another hull; against spheres / capsules / cylinders the fitted proxy stands in
  const bool ha = ia[5] > 0, hb_ = ib[5] > 0;
  if ((ha && (hb_ || tb == SHAPE_BOX)) || (hb_ && (ha || ta == SHAPE_BOX))) {
    Ct loc[16]; int nloc = 0;
    collide_convex(C, ia, fa, Ra, pa, ib, fb, Rb, pb, mu, margin, loc, &nloc);
    for (int i = 0; i < nloc; i++) for (int j = i + 1; j < nloc; j++) if (loc[j].dist < loc[i].dist) { Ct t = loc[i]; loc[i] = loc[j]; loc[j] = t; }
    if (nloc > 4) nloc = 4;
    for (int i = 0; i < nloc; i++) out[nt_++] = loc[i];
    return nt_;
  }
  if (ta != SHAPE_BOX && tb != SHAPE_BOX) {
    float a0[3], a1[3], b0[3], b1[3], ra, rb, d1[3], d2[3], s, t, c1[3], c2[3];
    as_capsule(ta, fa + 7, Ra, pa, a0, a1, &ra); as_capsule(tb, fb + 7, Rb, pb, b0, b1, &rb);
    v_sub(d1, a1, a0); v_sub(d2, b1, b0); seg_closest(a0, d1, b0, d2, &s, &t);
    v_cpy(c1, a0); v_madd(c1, d1, s); v_cpy(c2, b0); v_madd(c2, d2, t);
    float d[3]; v_sub(d, c1, c2); float len = v_len(d);
    if (len < 1e-12f) v_set(n, 0, 0, 1); else v_scale(n, d, 1.0f / len);
    dist = len - ra - rb; float tt[3]; v_scale(tt, n, -ra); v_add(ca, c1, tt); v_scale(tt, n, rb); v_add(cb, c2, tt);
    ct_add(out, &nt_, 4, ia[1], ib[1], ca, cb, n, dist, mu, margin);
    return nt_;
  }
  // at least one box: B is the reference box, X the other shape (flip at the end if we swapped)
  int swap = (tb != SHAPE_BOX);
  const float *Rx = swap ? Rb : Ra, *px = swap ? pb : pa, *dx = swap ? fb + 7 : fa + 7;
  const float *Rbx = swap ? Ra : Rb, *pbx = swap ? pa : pb, *hb = swap ? fa + 7 : fb + 7;
  int tx = swap ? tb : ta; int fx = swap ? ib[1] : ia[1], fbx = swap ? ia[1] : ib[1];
  Ct loc[16]; int nloc = 0;
  if (tx == SHAPE_SPHERE) {
    if (sphere_box(px, dx[0], Rbx, pbx, hb, ca, cb, n, &dist)) ct_add(loc, &nloc, 16, fx, fbx, ca, cb, n, dist, mu, margin);
  } else if (tx == SHAPE_CAPSULE) {
    float e0[3], e1[3], rad, mid[3], dseg[3], rel[3];
    as_capsule(tx, dx, Rx, px, e0, e1, &rad);
    v_sub(dseg, e1, e0); v_sub(rel, pbx, e0);
    float dd = v_dot(dseg, dseg), tt = dd > 1e-18f ? clampf(v_dot(rel, dseg) / dd, 0.f, 1.f) : 0.0f;
    v_cpy(mid, e0); v_madd(mid, dseg, tt);
    if (sphere_box(e0, rad, Rbx, pbx, hb, ca, cb, n, &dist)) ct_add(loc, &nloc, 16, fx, fbx, ca, cb, n, dist, mu, margin);
    if (dd > 1e-18f && sphere_box(e1, rad, Rbx, pbx, hb, ca, cb, n, &dist)) ct_add(loc, &nloc, 16, fx, fbx, ca, cb, n, dist, mu, margin);
    if (tt > 1e-6f && tt < 1 - 1e-6f && sphere_box(mid, rad, Rbx, pbx, hb, ca, cb, n, &dist)) ct_add(loc, &nloc, 16, fx, fbx, ca, cb, n, dist, mu, margin);
  } else if (tx == SHAPE_CYLINDER) {
    float zc[3] = {Rx[2], Rx[5], Rx[8]}, xc[3] = {Rx[0], Rx[3], Rx[6]}, yc[3] = {Rx[1], Rx[4], Rx[7]};
    for (int cap = -1; cap <= 1; cap += 2) {
      float cc[3]; v_cpy(cc, px); v_madd(cc, zc, cap * dx[1]);
      for (int k = 0; k < 6; k++) {
        float sg = k < 3 ? 1.f : -1.f; int a3 = k % 3;
        float nk[3] = {-Rbx[a3] * sg, -Rbx[3 + a3] * sg, -Rbx[6 + a3] * sg};
        float t[3]; v_cpy(t, nk); v_madd(t, zc, -v_dot(nk, zc));
        float len = v_len(t), pt[3];
        int npt = len < 1e-6f ? 4 : 1;   // cap parallel to this face: four rim points instead
        for (int j4 = 0; j4 < npt; j4++) {
          if (npt == 4) { const float* bx = (j4 & 1) ? yc : xc; float s2 = (j4 & 2) ? -1.0f : 1.0f; v_cpy(pt, cc); v_madd(pt, bx, s2 * dx[0]); }
          else { v_cpy(pt, cc); v_madd(pt, t, dx[0] / len); }
          if (point_box(pt, Rbx, pbx, hb, margin, cb, n, &dist)) {
            int dup = 0;
            for (int j = 0; j < nloc; j++) { float dd[3]; v_sub(dd, loc[j].pa, pt); if (v_dot(dd, dd) < 1e-12f) dup = 1; }
            if (!dup) ct_add(loc, &nloc, 16, fx, fbx, pt, cb, n, dist, mu, margin);
          }
        }
      }
    }
  } else {   // box X against box B: corners of X in B, then corners of B in X
    for (int k = 0; k < 8; k++) {
      float cl[3] = {(k & 1 ? 1 : -1) * dx[0], (k & 2 ? 1 : -1) * dx[1], (k & 4 ? 1 : -1) * dx[2]}, pt[3], t[3];
      m_vec(t, Rx, cl); v_add(pt, px, t);
      if (point_box(pt, Rbx, pbx, hb, margin, cb, n, &dist)) ct_add(loc, &nloc, 16, fx, fbx, pt, cb, n, dist, mu, margin);
    }
    for (int k = 0; k < 8; k++) {
      float cl[3] = {(k & 1 ? 1 : -1) * hb[0], (k & 2 ? 1 : -1) * hb[1], (k & 4 ? 1 : -1) * hb[2]}, pt[3], t[3], nn[3], cx[3];
      m_vec(t, Rbx, cl); v_add(pt, pbx, t);
      if (point_box(pt, Rx, px, dx, margin, cx, nn, &dist)) { v_scale(nn, nn, -1.0f); ct_add(loc, &nloc, 16, fx, fbx, cx, pt, nn, dist, mu, margin); }
    }
  }
  // keep the 4 deepest (stable selection, same order as a stable sort by depth)
  for (int i = 0; i < nloc; i++) for (int j = i + 1; j < nloc; j++) if (loc[j].dist < loc[i].dist) { Ct t = loc[i]; loc[i] = loc[j]; loc[j] = t; }
  if (nloc > 4) nloc = 4;
  for (int i = 0; i < nloc; i++) {
    Ct c = loc[i];
    if (swap) { Ct s2 = c; s2.fa = c.fb; s2.fb = c.fa; v_cpy(s2.pa, c.pb); v_cpy(s2.pb, c.pa); v_scale(s2.n, c.n, -1.0f); c = s2; }
    out[nt_++] = c;
  }
  return nt_;
}
DG_HD void surv_set(int* word, int bit) {
#if defined(__CUDA_ARCH__)
  atomicOr(word, 1 << bit);
#else
  *word |= 1 << bit;
#endif
}
DG_HD int ffs64(unsigned long long x) {
#if defined(__CUDA_ARCH__)
  return __ffsll((long long)x);
#else
  return __builtin_ffsll((long long)x);
#endif
}
DG_HD int popc32(unsigned x) {
#if defined(__CUDA_ARCH__)
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}
// broad phase: bounding-sphere test of every candidate pair, survivors marked in a bit set
DG_FN void phase_broad(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  for (int it = ln; it < sc.ngrp + sc.nloose; it += nt) {
    if (it < sc.ngrp) {
      // one test of the static shape against the body's bounding sphere rules out the whole group
      const int* g = gc(sc.grp_i) + 4 * it; const float* w = gc(sc.shape_wb) + 12 * g[0];
      const float* cb = KIN(gc(sc.body_plan)[BP_W * g[1] + BP_SLOT]) + 9;
      float dc[3]; v_sub(dc, w + 9, cb);
      float reach = gc(sc.shape_f)[DG_SHAPE_F_W * g[0] + 11] + gc(sc.body_reach)[g[1]] + sc.margin;
      if (v_dot(dc, dc) > reach * reach) continue;
      {   // a static box (a maze wall, a table top) against the body's sphere: the box itself, not its bounding ball
        const int* is = gc(sc.shape_i) + DG_SHAPE_I_W * g[0];
        if (is[2] == SHAPE_BOX && is[5] == 0) {
          const float* h = gc(sc.shape_f) + DG_SHAPE_F_W * g[0] + 7;
          float d[3], pl[3]; v_sub(d, cb, w + 9); mT_vec(pl, w, d);
          float d2 = 0.f;
          for (int i = 0; i < 3; i++) { const float ex = fabsf(pl[i]) - h[i]; if (ex > 0.f) d2 += ex * ex; }
          const float r = gc(sc.body_reach)[g[1]] + sc.margin;
          if (d2 > r * r) continue;
        }
      }
      for (int j = 0; j < g[3]; j++) {
        int k = gc(sc.grp_pairs)[g[2] + j];
        if (pair_in_reach(C, gc(sc.pair_i)[2 * k], gc(sc.pair_i)[2 * k + 1])) surv_set(WSIP(C, sc.X_SURV) + (k >> 5), k & 31);
      }
    } else {
      int k = gc(sc.loose_pairs)[it - sc.ngrp];
      if (pair_in_reach(C, gc(sc.pair_i)[2 * k], gc(sc.pair_i)[2 * k + 1])) surv_set(WSIP(C, sc.X_SURV) + (k >> 5), k & 31);
    }
  }
}
DG_FN void phase_count_survivors(const Env& C, int ln, int nt) {
  if (ln != 0) return;
  int nw = (SC.npair + 31) / 32, n = 0;
  for (int i = 0; i < nw; i++) n += popc32((unsigned)WSIP(C, SC.X_SURV)[i]);
  WSI(C)[SC.W_HDR + WH_NSURV] = n;
}
// narrow phase, round `rnd`: lane ln takes survivor number rnd*nt + ln (in pair order) and parks its contacts
DG_FN void phase_narrow(const Env& C, int ln, int nt, int rnd) {
  const DevScene& sc = SC;
  float* tmp = WSG(C, sc.X_CTMP) + sc.ctmp_stride * ln;
  int want = rnd * nt + ln, nw = (sc.npair + 31) / 32, seen = 0, pair = -1;
  for (int i = 0; i < nw && pair < 0; i++) {
    unsigned wd = (unsigned)WSIP(C, sc.X_SURV)[i]; int c = popc32(wd);
    if (seen + c <= want) { seen += c; continue; }
    for (int bit = 0; bit < 32; bit++) if (wd & (1u << bit)) { if (seen == want) { pair = 32 * i + bit; break; } seen++; }
  }
  int n = 0;
  if (pair >= 0) {
    Ct out[4];
    n = collide_pair(C, gc(sc.pair_i)[2 * pair], gc(sc.pair_i)[2 * pair + 1], out);
    for (int i = 0; i < n; i++) {
      float* c = tmp + 1 + CT_W * i;
      c[CT_FA] = int_as_float(out[i].fa); c[CT_FB] = int_as_float(out[i].fb);
      v_cpy(c + CT_PA, out[i].pa); v_cpy(c + CT_PB, out[i].pb); v_cpy(c + CT_N, out[i].n); c[CT_DIST] = out[i].dist; c[CT_MU] = out[i].mu;
    }
  }
  tmp[0] = int_as_float(n);
}
// Capacity max_contacts (YAML extension key; default 16 with a floating body, else 8, at most 21): when the list is full a
// new contact replaces the SHALLOWEST stored one if it is deeper - what gets lost is a grazing contact, never the wall the
// robot is pushing into - and every loss is counted (dg_query DG_Q_CONTACTS_DROPPED).  Same rule as the oracle.
DG_FN void phase_append(const Env& C, int ln, int nt) {
  if (ln != 0) return;
  const DevScene& sc = SC;
  int nc = WSI(C)[sc.W_HDR + WH_NCONTACT], lost = 0;
  for (int l = 0; l < nt; l++) {
    const float* tmp = WSG(C, sc.X_CTMP) + sc.ctmp_stride * l; int n = float_as_int(tmp[0]);
    for (int i = 0; i < n; i++) {
      const float* src = tmp + 1 + CT_W * i; float* dst;
      if (nc < sc.maxc) dst = WSP(C, sc.X_CON) + CT_W * nc++;
      else {
        lost++;
        int worst = 0; float wd = (WSP(C, sc.X_CON))[CT_DIST];
        for (int j = 1; j < nc; j++) { const float dj = (WSP(C, sc.X_CON) + CT_W * j)[CT_DIST]; if (dj > wd) { wd = dj; worst = j; } }
        if (nc == 0 || !(src[CT_DIST] < wd)) continue;
        dst = WSP(C, sc.X_CON) + CT_W * worst;
      }
      for (int j = 0; j < CT_W; j++) dst[j] = src[j];
    }
  }
  WSI(C)[sc.W_HDR + WH_NCONTACT] = nc;
  if (lost && C.dropped) {
#if defined(__CUDA_ARCH__)
    atomicAdd(C.dropped, (unsigned)lost);
#else
    *C.dropped += (unsigned)lost;
#endif
  }
}

// ------------------------------------------------------------------ constraint rows ----------------------------
DG_HD int body_of_frame(const Env& C, int f) { return f < C.sc->nb ? f : shc(C.link_i)[DG_LINK_I_W * (f - C.sc->nb)]; }
// generalized force per unit force along dir at world point p on frame f (compact coordinates of its body)
DG_FN void point_jacobian(const Env& C, int f, const float* p, const float* dir, float* J) {
  const DevScene& sc = SC;
  int b = body_of_frame(C, f); const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
  int g = bp[BP_GDIM], d0 = bi[3], s0 = bp[BP_SLOT], l0 = bi[1];
  for (int i = 0; i < g; i++) J[i] = 0.f;
  int jo = 0;
  if (bi[0] == 2) { float rel[3]; v_sub(rel, p, KIN(s0) + 9); v_cross(J, rel, dir); v_cpy(J + 3, dir); jo = 6; }
  int gl = f < sc.nb ? -1 : f - sc.nb;
  while (gl >= 0) {
    const int* li = shc(C.link_i) + DG_LINK_I_W * gl; const float* lf = shc(C.link_f) + DG_LINK_F_W * gl; const float* K = KIN(s0 + 1 + gl - l0);
    if (li[2] == 1) {
      float aw[3], dw[3], o[3], rel[3], t[3];
      m_vec(aw, K, lf + 10); m_vec(dw, K, lf + 7); v_sub(o, K + 9, dw);
      v_sub(rel, p, o); v_cross(t, aw, rel); J[jo + li[3] - d0] = v_dot(dir, t);
    } else if (li[2] == 2) { float aw[3]; m_vec(aw, K, lf + 10); J[jo + li[3] - d0] = v_dot(dir, aw); }
    gl = li[1];
  }
}
// generalized force per unit TORQUE along dir on frame f (compact coordinates of its body)
DG_FN void angular_jacobian(const Env& C, int f, const float* dir, float* J) {
  const DevScene& sc = SC;
  int b = body_of_frame(C, f); const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
  int g = bp[BP_GDIM], d0 = bi[3], s0 = bp[BP_SLOT], l0 = bi[1], jo = 0;
  for (int i = 0; i < g; i++) J[i] = 0.f;
  if (bi[0] == 2) { v_cpy(J, dir); jo = 6; }
  for (int gl = f < sc.nb ? -1 : f - sc.nb; gl >= 0; gl = shc(C.link_i)[DG_LINK_I_W * gl + 1]) {
    const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
    if (li[2] == 1) { float aw[3]; m_vec(aw, KIN(s0 + 1 + gl - l0), shc(C.link_f) + DG_LINK_F_W * gl + 10); J[jo + li[3] - d0] = v_dot(dir, aw); }
  }
}
DG_FN void body_genvel(const Env& C, int b, float* gv) {
  const int* bi = gc(SC.body_i) + DG_BODY_I_W * b; int jo = 0;
  if (bi[0] == 2) { const float* bs = BST(gc(SC.body_plan)[BP_W * b + BP_DI]); v_cpy(gv, bs + 10); v_cpy(gv + 3, bs + 7); jo = 6; }
  for (int i = 0; i < bi[4]; i++) gv[jo + i] = DOF(D_QD, bi[3] + i);
}
// joint-limit rows (only when violated) then motor rows of every dynamic body, lane per body
DG_FN void phase_unit_rows(const Env& C, int ln, int nt, float h) {
  const DevScene& sc = SC;
  for (int di = ln; di < sc.ndyn; di += nt) {
    int b = gc(sc.dyn_body)[di]; const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
    int l0 = bi[1], nlb = bi[2], d0 = bi[3], g = bp[BP_GDIM], gs = bp[BP_GS], jo = bi[0] == 2 ? 6 : 0;
    const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF];
    float* rows = WSH(C, sc.X_UROW) + UR_W * bp[BP_UROW]; int n = 0;
    for (int k = 0; k < nlb; k++) {
      const int* li = shc(C.link_i) + DG_LINK_I_W * (l0 + k); const float* lf = shc(C.link_f) + DG_LINK_F_W * (l0 + k);
      int d = li[3];
      if (d < 0 || !li[4]) continue;
      for (int side = 0; side < 2; side++) {
        float pen = side == 0 ? DOF(D_Q, d) - lf[20] : lf[21] - DOF(D_Q, d);
        if (pen > 0) continue;
        int col = jo + d - d0; float sg = side == 0 ? 1.f : -1.f;
        float den = Minv[col * gs + col], dinv = den > 1e-30f ? 1.0f / den : 0.f, rel = sg * DOF(D_QD, d);
        float* r = rows + UR_W * n++;
        r[UR_RHS] = (-rel + (-pen) * sc.erp / h) * dinv; r[UR_DINV] = dinv; r[UR_LO] = 0.f; r[UR_HI] = sc.limit_max_impulse; r[UR_APPLIED] = 0.f;
        r[UR_COL] = int_as_float(side == 0 ? col : -1 - col); r[UR_MOTOR] = int_as_float(-1);
      }
    }
    for (int k = 0; k < nlb; k++) {
      int d = shc(C.link_i)[DG_LINK_I_W * (l0 + k) + 3];
      if (d < 0) continue;
      float maxf = ST(S_MMAXF)[d];
      DOF(D_APPLIED, d) = 0.f;
      if (maxf <= 0) continue;
      int col = jo + d - d0;
      float den = Minv[col * gs + col], dinv = den > 1e-30f ? 1.0f / den : 0.f, qd = DOF(D_QD, d);
      float desired = ST(S_MKP)[d] * (ST(S_MTPOS)[d] - DOF(D_Q, d)) / h + qd + ST(S_MKD)[d] * (ST(S_MTVEL)[d] - qd);
      float* r = rows + UR_W * n++;
      r[UR_RHS] = (desired - qd) * dinv; r[UR_DINV] = dinv; const float cdt = (sc.sem & SEM_MOTOR_CLAMP_SUBSTEP) ? h : sc.dt;   // impulse clamp: max force x outer dt (default) or x sub-step dt
      r[UR_LO] = -maxf * cdt; r[UR_HI] = maxf * cdt; r[UR_APPLIED] = 0.f;
      r[UR_COL] = int_as_float(col); r[UR_MOTOR] = int_as_float(d);
    }
    WSI(C)[sc.W_UCNT + di] = n;
    float* dv = WSH(C, sc.W_DV) + bp[BP_GVOFF];
    for (int i = 0; i < gs; i++) dv[i] = 0.f;
    // row-space system A[r][s] = J_r M^-1 J_s^T for the register-resident sweep (pgs_unit_fast)
    int nrs = bp[BP_NRS];
    if (n <= nrs) {
      float* A = WSH(C, sc.X_AMAT) + bp[BP_AOFF];
      for (int r = 0; r < n; r++) {
        int cr = float_as_int(rows[UR_W * r + UR_COL]); float sr = 1.f; if (cr < 0) { cr = -1 - cr; sr = -1.f; }
        for (int s2 = 0; s2 < nrs; s2++) {
          float a = 0.f;
          if (s2 < n) { int cs = float_as_int(rows[UR_W * s2 + UR_COL]); float ss = 1.f; if (cs < 0) { cs = -1 - cs; ss = -1.f; } a = sr * ss * Minv[cr * gs + cs]; }
          A[r * nrs + s2] = a;
        }
      }
    }
  }
  if (ln == 0) { WSI(C)[sc.W_HDR + WH_NCROW] = 3 * WSI(C)[sc.W_HDR + WH_NCONTACT]; WSI(C)[sc.W_HDR + WH_COUPLED] = 0; }
}
DG_FN void plane_space(const float* n, float* p, float* q) {
  if (fabsf(n[2]) > 0.7071067811865475244f) { float a = n[1] * n[1] + n[2] * n[2], k = 1.0f / sqrtf(a); p[0] = 0; p[1] = -n[2] * k; p[2] = n[1] * k; q[0] = a * k; q[1] = -n[0] * p[2]; q[2] = n[0] * p[1]; }
  else { float a = n[0] * n[0] + n[1] * n[1], k = 1.0f / sqrtf(a); p[0] = -n[1] * k; p[1] = n[0] * k; p[2] = 0; q[0] = -n[2] * p[1]; q[1] = n[2] * p[0]; q[2] = a * k; }
}
// contact rows: normals [0, nc), then two friction rows per contact; lane per row
DG_FN void phase_contact_rows(const Env& C, int ln, int nt, float h) {
  const DevScene& sc = SC;
  int nc = WSI(C)[sc.W_HDR + WH_NCONTACT];
  for (int r = ln; r < 3 * nc; r += nt) {
    int k = r < nc ? r : (r - nc) >> 1, dirk = r < nc ? -1 : (r - nc) & 1;
    const float* c = WSP(C, sc.X_CON) + CT_W * k;
    int fa = float_as_int(c[CT_FA]), fb = float_as_int(c[CT_FB]);
    float dir[3];
    if (dirk < 0) v_cpy(dir, c + CT_N); else { float t1[3], t2[3]; plane_space(c + CT_N, t1, t2); v_cpy(dir, dirk == 0 ? t1 : t2); }
    float* row = WSP(C, sc.X_CROW) + sc.crow_stride * r; float* J = row + CR_HDR; float* M = J + sc.GP;
    int ba = body_of_frame(C, fa), bb = body_of_frame(C, fb);
    int dia = gc(sc.body_plan)[BP_W * ba + BP_DI], dib = gc(sc.body_plan)[BP_W * bb + BP_DI];
    float den = 0.f, rel = 0.f; int ga = 0;
    if (dia >= 0) {
      const int* bp = gc(sc.body_plan) + BP_W * ba; ga = bp[BP_GDIM]; const int gsa = bp[BP_GS]; const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF];
      point_jacobian(C, fa, c + CT_PA, dir, J);
      body_genvel(C, ba, M);   // M doubles as scratch for the generalized velocity
      for (int i = 0; i < ga; i++) rel += J[i] * M[i];
      for (int i = 0; i < ga; i++) { float s = 0.f; for (int j = 0; j < ga; j++) s += Minv[j * gsa + i] * J[j]; M[i] = s; }
      for (int i = 0; i < ga; i++) den += J[i] * M[i];
    }
    if (dib >= 0) {
      const int* bp = gc(sc.body_plan) + BP_W * bb; int gb = bp[BP_GDIM]; const int gsb = bp[BP_GS]; const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF];
      float nd_[3]; v_scale(nd_, dir, -1.0f);
      float *JB = J + ga, *MB = M + ga;
      point_jacobian(C, fb, c + CT_PB, nd_, JB);
      body_genvel(C, bb, MB);
      for (int i = 0; i < gb; i++) rel += JB[i] * MB[i];
      for (int i = 0; i < gb; i++) { float s = 0.f; for (int j = 0; j < gb; j++) s += Minv[j * gsb + i] * JB[j]; MB[i] = s; }
      for (int i = 0; i < gb; i++) den += JB[i] * MB[i];
    }
    { int used = ga + (dib >= 0 ? gc(sc.body_plan)[BP_W * bb + BP_GDIM] : 0); for (int i = used; i < sc.GP; i++) { J[i] = 0.f; M[i] = 0.f; } }
    if (dia >= 0 && dib >= 0) WSI(C)[sc.W_HDR + WH_COUPLED] = 1;   // a row couples two dynamic bodies: lock-step sweeps needed
    float dinv = den > 1e-30f ? 1.0f / den : 0.f;
    row[CR_DINV] = dinv; row[CR_APPLIED] = 0.f; row[CR_MU] = c[CT_MU]; WSH(C, sc.W_CAPP)[r] = 0.f;
    row[CR_DA] = int_as_float(dia); row[CR_DB] = int_as_float(dib);
    if (dirk < 0) {
      float pen = c[CT_DIST] + sc.slop, pos_err = 0.f, vel_err = -rel;
      if (pen > 0) vel_err -= pen / h; else pos_err = -pen * sc.cerp / h;
      row[CR_RHS] = (pos_err + vel_err) * dinv; row[CR_LO] = 0.f; row[CR_HI] = 1e10f; row[CR_PARENT] = int_as_float(-1);
    } else {
      row[CR_RHS] = -rel * dinv; row[CR_LO] = 0.f; row[CR_HI] = 0.f; row[CR_PARENT] = int_as_float(k);
    }
  }
}

// ------------------------------------------------------------------ projected Gauss-Seidel ---------------------
DG_FN void pgs_unit_sweep(const Env& C, int b, int di, int it) {
  const DevScene& sc = SC;
  const int* bp = gc(sc.body_plan) + BP_W * b; int g = bp[BP_GDIM], gs = bp[BP_GS], n = WSI(C)[sc.W_UCNT + di];
  const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF]; float* dv = WSH(C, sc.W_DV) + bp[BP_GVOFF];
  float* rows = WSH(C, sc.X_UROW) + UR_W * bp[BP_UROW];
  for (int j = 0; j < n; j++) {
    float* r = rows + UR_W * ((it & 1) ? j : n - 1 - j);
    int colc = float_as_int(r[UR_COL]); float sg = 1.f; int col = colc;
    if (colc < 0) { col = -1 - colc; sg = -1.f; }
    float d = r[UR_RHS] - sg * dv[col] * r[UR_DINV];
    float ap = r[UR_APPLIED], sum = ap + d, lo = r[UR_LO], hi = r[UR_HI];
    if (sum < lo) { d = lo - ap; sum = lo; } else if (sum > hi) { d = hi - ap; sum = hi; }
    r[UR_APPLIED] = sum;
    float sd = sg * d; const float* Mc = Minv + col * gs;
    for (int i = 0; i < g; i++) dv[i] = fmaf(Mc[i], sd, dv[i]);
  }
}
// Register-resident sweeps over the unit rows of one body, iterations [it0, it1): same Gauss-Seidel order and
// clamps as pgs_unit_sweep, carried out in row space (y_r = J_r dv) so that every index is a compile-time constant.
// NR >= number of rows; the padding rows carry zeros (rhs = dinv = lo = hi = 0, zero A row) and change nothing.
// For NR <= 8 the row-space matrix A lives in registers as well, so the 150 sweeps touch no memory at all.
template <int NR>
DG_FN void pgs_unit_fast(const Env& C, int b, int di, int it0, int it1) {
  const DevScene& sc = SC;
  const int* bp = gc(sc.body_plan) + BP_W * b; const int g = bp[BP_GDIM], gs = bp[BP_GS], nrs = bp[BP_NRS], n = WSI(C)[sc.W_UCNT + di];
  const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF]; float* dv = WSH(C, sc.W_DV) + bp[BP_GVOFF];
  float* rows = WSH(C, sc.X_UROW) + UR_W * bp[BP_UROW]; const float* A = WSH(C, sc.X_AMAT) + bp[BP_AOFF];
  constexpr bool kRegA = NR <= 8;
  float rhs[NR], dinv[NR], lo[NR], hi[NR], ap[NR], ap0[NR], y[NR], Ar[kRegA ? NR * NR : 1];
#pragma unroll
  for (int r = 0; r < NR; r++) {
    rhs[r] = 0.f; dinv[r] = 0.f; lo[r] = 0.f; hi[r] = 0.f; ap[r] = 0.f; y[r] = 0.f;
    if (r < n) {
      const float* rw = rows + UR_W * r;
      rhs[r] = rw[UR_RHS]; dinv[r] = rw[UR_DINV]; lo[r] = rw[UR_LO]; hi[r] = rw[UR_HI]; ap[r] = rw[UR_APPLIED];
      int c = float_as_int(rw[UR_COL]);
      y[r] = c < 0 ? -dv[-1 - c] : dv[c];
    }
    ap0[r] = ap[r];
    if (kRegA) {
#pragma unroll
      for (int s2 = 0; s2 < NR; s2++) Ar[kRegA ? r * NR + s2 : 0] = (r < n && s2 < n) ? A[r * nrs + s2] : 0.f;
    }
  }
#define DG_PGS_ROW(r)                                                                        \
  {                                                                                          \
    float d = rhs[r] - y[r] * dinv[r];                                                       \
    float sum = ap[r] + d;                                                                   \
    const bool below = sum < lo[r], above = sum > hi[r];                                     \
    d = below ? lo[r] - ap[r] : (above ? hi[r] - ap[r] : d);                                 \
    ap[r] = below ? lo[r] : (above ? hi[r] : sum);                                           \
    if (kRegA) {                                                                             \
      _Pragma("unroll") for (int s2 = 0; s2 < NR; s2++) y[s2] = fmaf(Ar[kRegA ? (r) * NR + s2 : 0], d, y[s2]); \
    } else if ((r) < n) {                                                                    \
      const float* Am = A + (r) * nrs;                                                       \
      _Pragma("unroll") for (int s2 = 0; s2 < NR; s2++) y[s2] = fmaf(Am[s2], d, y[s2]);      \
    }                                                                                        \
  }
  for (int it = it0; it < it1; it++) {
    if (it & 1) {
#pragma unroll
      for (int r = 0; r < NR; r++) DG_PGS_ROW(r)
    } else {
#pragma unroll
      for (int r = NR - 1; r >= 0; r--) DG_PGS_ROW(r)
    }
  }
#undef DG_PGS_ROW
#pragma unroll
  for (int r = 0; r < NR; r++) if (r < n) {
    float* rw = rows + UR_W * r;
    rw[UR_APPLIED] = ap[r];
    float dl = ap[r] - ap0[r];
    int c = float_as_int(rw[UR_COL]); if (c < 0) { c = -1 - c; dl = -dl; }
    const float* Mc = Minv + c * gs;
    for (int i = 0; i < g; i++) dv[i] = fmaf(Mc[i], dl, dv[i]);
  }
}
DG_FN void pgs_unit_any(const Env& C, int b, int di, int it0, int it1) {
  const int nrs = gc(SC.body_plan)[BP_W * b + BP_NRS], n = WSI(C)[SC.W_UCNT + di];
  if (n == 0) return;
  if (n <= nrs) {   // the A matrix was built (phase_unit_rows); nrs is a multiple of 4, so the padded reads stay inside it
    if (n <= 4) { pgs_unit_fast<4>(C, b, di, it0, it1); return; }
    if (n <= 6 && nrs >= 8) { pgs_unit_fast<6>(C, b, di, it0, it1); return; }
    if (n <= 8) { pgs_unit_fast<8>(C, b, di, it0, it1); return; }
    if (n <= 12) { pgs_unit_fast<12>(C, b, di, it0, it1); return; }
    if (n <= 16) { pgs_unit_fast<16>(C, b, di, it0, it1); return; }
  }
  for (int it = it0; it < it1; it++) pgs_unit_sweep(C, b, di, it);
}
// All solver sweeps of ONE body whose contact rows touch no other dynamic body: unit rows then its contact rows,
// every iteration, with the generalized velocity change dv held in registers (G >= padded coordinate count).
template <int G>
DG_FN void pgs_body_full(const Env& C, int b, int di) {
  const DevScene& sc = SC;
  const int* bp = gc(sc.body_plan) + BP_W * b; const int gs = bp[BP_GS], n = WSI(C)[sc.W_UCNT + di];
  const int ncr = WSI(C)[sc.W_HDR + WH_NCROW];
  const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF]; float* dvs = WSH(C, sc.W_DV) + bp[BP_GVOFF];
  float* rows = WSH(C, sc.X_UROW) + UR_W * bp[BP_UROW];
  float* capp = WSH(C, sc.W_CAPP);
  unsigned long long mine = 0ull;   // the contact rows that act on this body (at most 63 rows: max_contacts <= 21)
  for (int rr = 0; rr < ncr && rr < 63; rr++) {
    const float* row = WSP(C, sc.X_CROW) + sc.crow_stride * rr;
    if (float_as_int(row[CR_DA]) == di || float_as_int(row[CR_DB]) == di) mine |= 1ull << rr;
  }
  float dv[G];
#pragma unroll
  for (int i = 0; i < G; i++) dv[i] = 0.f;
  for (int it = 0; it < sc.iters; it++) {
    for (int j = 0; j < n; j++) {
      float* r = rows + UR_W * ((it & 1) ? j : n - 1 - j);
      int col = float_as_int(r[UR_COL]); float sg = 1.f;
      if (col < 0) { col = -1 - col; sg = -1.f; }
      float x = 0.f;
#pragma unroll
      for (int i = 0; i < G; i++) x = (i == col) ? dv[i] : x;
      float d = r[UR_RHS] - sg * x * r[UR_DINV];
      float ap = r[UR_APPLIED], sum = ap + d, lo = r[UR_LO], hi = r[UR_HI];
      if (sum < lo) { d = lo - ap; sum = lo; } else if (sum > hi) { d = hi - ap; sum = hi; }
      r[UR_APPLIED] = sum;
      float sd = sg * d; const float* Mc = Minv + col * gs;
#pragma unroll
      for (int c4 = 0; c4 < G / 4; c4++) if (4 * c4 < gs) {
        F4 m = ld4(Mc + 4 * c4);
        dv[4 * c4] = fmaf(m.x, sd, dv[4 * c4]); dv[4 * c4 + 1] = fmaf(m.y, sd, dv[4 * c4 + 1]);
        dv[4 * c4 + 2] = fmaf(m.z, sd, dv[4 * c4 + 2]); dv[4 * c4 + 3] = fmaf(m.w, sd, dv[4 * c4 + 3]);
      }
    }
    for (unsigned long long m = mine; m != 0ull; m &= m - 1ull) {
      const int rr = ffs64(m) - 1;
      const float* row = WSP(C, sc.X_CROW) + sc.crow_stride * rr;
      const float* J = row + CR_HDR; const float* M = J + sc.GP;
      // every load of the row is issued before the first use (one memory round trip per row instead of three)
      const F4 h = ld4(row), h2 = ld4(row + 4), h3 = ld4(row + 8);   // rhs dinv lo hi | - mu da db | parent
      F4 jv[G / 4], mv[G / 4];
#pragma unroll
      for (int c4 = 0; c4 < G / 4; c4++) {
        if (4 * c4 < gs) { jv[c4] = ld4(J + 4 * c4); mv[c4] = ld4(M + 4 * c4); }
        else { F4 z = {0.f, 0.f, 0.f, 0.f}; jv[c4] = z; mv[c4] = z; }
      }
      float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
      for (int c4 = 0; c4 < G / 4; c4++) {
        d0 = fmaf(jv[c4].x, dv[4 * c4], d0); d1 = fmaf(jv[c4].y, dv[4 * c4 + 1], d1); d2 = fmaf(jv[c4].z, dv[4 * c4 + 2], d2); d3 = fmaf(jv[c4].w, dv[4 * c4 + 3], d3);
      }
      float d = h.x - ((d0 + d1) + (d2 + d3)) * h.y;
      float lo = h.z, hi = h.w;
      const int par = float_as_int(h3.x);
      if (par >= 0) { hi = h2.y * capp[par]; lo = -hi; }
      const float ap = capp[rr]; float sum = ap + d;
      const bool below = sum < lo, above = sum > hi;
      d = below ? lo - ap : (above ? hi - ap : d);
      capp[rr] = below ? lo : (above ? hi : sum);
#pragma unroll
      for (int c4 = 0; c4 < G / 4; c4++) {
        dv[4 * c4] = fmaf(mv[c4].x, d, dv[4 * c4]); dv[4 * c4 + 1] = fmaf(mv[c4].y, d, dv[4 * c4 + 1]);
        dv[4 * c4 + 2] = fmaf(mv[c4].z, d, dv[4 * c4 + 2]); dv[4 * c4 + 3] = fmaf(mv[c4].w, d, dv[4 * c4 + 3]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < G; i++) if (i < gs) dvs[i] = dv[i];
}
DG_FN void phase_pgs_full(const Env& C, int ln, int nt) {
  for (int di = ln; di < SC.ndyn; di += nt) {
    int b = gc(SC.dyn_body)[di], gs = gc(SC.body_plan)[BP_W * b + BP_GS];
    if (gs <= 8) pgs_body_full<8>(C, b, di); else if (gs <= 16) pgs_body_full<16>(C, b, di); else pgs_body_full<32>(C, b, di);
  }
}
DG_FN void pgs_contact_sweep(const Env& C) {
  const DevScene& sc = SC;
  int ncr = WSI(C)[sc.W_HDR + WH_NCROW];
  for (int r = 0; r < ncr; r++) {
    float* row = WSP(C, sc.X_CROW) + sc.crow_stride * r; const float* J = row + CR_HDR; const float* M = J + sc.GP;
    int dia = float_as_int(row[CR_DA]), dib = float_as_int(row[CR_DB]);
    float dot = 0.f; int ga = 0; float *dva = nullptr, *dvb = nullptr; int gb = 0;
    if (dia >= 0) { const int* bp = gc(sc.body_plan) + BP_W * gc(sc.dyn_body)[dia]; ga = bp[BP_GDIM]; dva = WSH(C, sc.W_DV) + bp[BP_GVOFF]; for (int i = 0; i < ga; i++) dot += J[i] * dva[i]; }
    if (dib >= 0) { const int* bp = gc(sc.body_plan) + BP_W * gc(sc.dyn_body)[dib]; gb = bp[BP_GDIM]; dvb = WSH(C, sc.W_DV) + bp[BP_GVOFF]; for (int i = 0; i < gb; i++) dot += J[ga + i] * dvb[i]; }
    float d = row[CR_RHS] - dot * row[CR_DINV];
    float lo = row[CR_LO], hi = row[CR_HI];
    int par = float_as_int(row[CR_PARENT]);
    float* capp = WSH(C, sc.W_CAPP);
    if (par >= 0) { hi = row[CR_MU] * capp[par]; lo = -hi; }
    float ap = capp[r], sum = ap + d;
    if (sum < lo) { d = lo - ap; sum = lo; } else if (sum > hi) { d = hi - ap; sum = hi; }
    capp[r] = sum;
    for (int i = 0; i < ga; i++) dva[i] = fmaf(M[i], d, dva[i]);
    for (int i = 0; i < gb; i++) dvb[i] = fmaf(M[ga + i], d, dvb[i]);
  }
}
DG_FN void phase_pgs_unit(const Env& C, int ln, int nt, int it0, int it1) {
  for (int di = ln; di < SC.ndyn; di += nt) pgs_unit_any(C, gc(SC.dyn_body)[di], di, it0, it1);
}
DG_FN void phase_pgs_contact(const Env& C, int ln, int nt) { if (ln == 0) pgs_contact_sweep(C); }
// ------------------------------------------------------------------ row-space team solver ----------------------
// Environments with contacts (or welded models) are solved by the WHOLE team in row space: y_p = J_p dv is carried for
// every unit, constraint and contact row, A[p][s] = J_s M^-1 J_p^T is built once per sub-step by all lanes, and one
// Gauss-Seidel update of row p is  d = clamp(rhs_p - y_p dinv_p),  y_s += A[p][s] d.  Row order, clamps and friction bounds
// are those of the dv-space sweeps (pgs_body_full / pgs_contact_sweep) and of the oracle: unit rows (direction alternating
// with the iteration), constraint + normal rows, friction rows bounded by mu x (normal impulse after this sweep's normal
// rows).  Rows that couple two dynamic bodies need no special case: their A entries simply have two body terms.
//
// Layout.  Rows live at POSITIONS of three sections, each padded to a multiple of K (K = 2, 4 or 8 rows per lane):
//   [0, nu) unit rows | [P1, P1 + nk) constraint rows, [P1 + nk, P1 + nk + nc) normals | [P2, P2 + 2 nc) friction rows,
//   P1 = pad(nu), P2 = P1 + pad(nk + nc), Rp = P2 + pad(2 nc).
// A padding position carries rhs = dinv = lo = hi = 0 and a zero row / column of A: its update is d = 0 by arithmetic, no
// mask needed.  Lane l of the team OWNS positions [l K, (l + 1) K) - a BLOCK of consecutive rows - and keeps their y, rhs,
// clamps and accumulated impulses in registers; a sweep walks the blocks of a section in order, the K slots of a block
// unrolled.  Because consecutive rows belong to the same lane, the Gauss-Seidel dependency d_p -> y_{p+1} stays inside one
// thread (clamp + one FMA, ~25 cycles); the other lanes receive d_p by a shuffle whose latency is hidden - they fold it into
// their y one slot later - and only at a block boundary (every K rows) does the next owner wait for the broadcast.
// (Round 1 dealt the rows round-robin: every update then waited for a shuffle, ~270 cycles per row measured.)
// Setup scatters every row's J and M^-1 J^T into DENSE vectors over the generalized coordinates of all dynamic bodies
// (the layout of W_DV), so that building A and folding the impulses back into dv are plain dense products.
// home of A: the cold workspace (L1 / L2 backed).
struct RsLayout { int K, nu, nk, nc, P1, nrm0, nrm1, P2, fr1, Rp; };
DG_HD int rs_pad(int n, int K) { return (n + K - 1) / K * K; }
DG_HD int rs_total(int nu, int nk, int nc, int K) { return rs_pad(nu, K) + rs_pad(nk + nc, K) + rs_pad(2 * nc, K); }
DG_HD RsLayout rs_layout(int K, int nu, int nk, int nc) {
  RsLayout L; L.K = K; L.nu = nu; L.nk = nk; L.nc = nc; L.P1 = rs_pad(nu, K); L.nrm0 = L.P1 + nk; L.nrm1 = L.nrm0 + nc;
  L.P2 = L.P1 + rs_pad(nk + nc, K); L.fr1 = L.P2 + 2 * nc; L.Rp = L.P2 + rs_pad(2 * nc, K);
  return L;
}
DG_HD bool rs_real(const RsLayout& L, int p) { return p < L.nu || (p >= L.P1 && p < L.nrm1) || (p >= L.P2 && p < L.fr1); }
DG_FN RsLayout rs_layout_of(const Env& C) {
  const int* hdr = WSI(C) + SC.W_HDR;
  return rs_layout(hdr[WH_RS_K], hdr[WH_RS_NU], 6 * SC.ncons, hdr[WH_NCROW] / 3);
}
// smallest K whose padded layout fits a team of nt lanes (and the row capacity of the workspace); 0: does not fit
DG_HD int rs_kneed(int nu, int nk, int nc, int nt, int cap) {
  for (int K = 2; K <= RS_KMAX; K *= 2) { const int t = rs_total(nu, nk, nc, K); if (t <= K * nt && t <= cap) return K; }
  return 0;
}
// lane 0: row counts and the K this environment needs; WH_RS_NEED = 0 sends the environment to the dv-space sweeps
// (no contact, one-lane team, too many rows or coordinates)
DG_FN void phase_rs_plan(const Env& C, int ln, int nt) {
  if (ln != 0) return;
  const DevScene& sc = SC;
  int* hdr = WSI(C) + sc.W_HDR; const int ncr = hdr[WH_NCROW];
  int nu = 0;
  for (int di = 0; di < sc.ndyn; di++) nu += WSI(C)[sc.W_UCNT + di];
  const int nk = 6 * sc.ncons, nc = ncr / 3;
  const bool want = sc.solver == 1 && nt >= 2 && (nk > 0 || (ncr > 0 && (hdr[WH_COUPLED] != 0 || ncr >= sc.rs_min)));
  hdr[WH_RS_NU] = nu; hdr[WH_RS_R] = 0; hdr[WH_RS_DEFER] = 0;
  int need = want ? rs_kneed(nu, nk, nc, nt, sc.rs_cap) : 0;
  if (want && C.split) {
    // the sweep kernel gives an environment 8, 16 or 32 lanes with 4, 3 or 2 consecutive rows each (DevScene::rs_cls_*): the first
    // class whose K-padded layout fits; WH_RS_DEFER = 1 + class names the list, WH_RS_NEED the K of its layout
    for (int c = 0; c < RS_NCLS; c++) {
      const int kc = sc.rs_cls_k[c], rc = sc.rs_cls_r[c];
      if (rc <= 0) continue;
      const int t = rs_total(nu, nk, nc, kc);
      if (t <= rc && t <= sc.rs_cap) { need = kc; hdr[WH_RS_DEFER] = c + 1; break; }
    }
  }
  hdr[WH_RS_NEED] = need;
}
// row records + dense vectors, lane per row.  K is the largest need among the environments that share a warp in the sweeps
// (C.grp0 .. C.grp1: their workspaces sit at multiples of w_total from this one), so that the warp runs one instantiation.
DG_FN void phase_rs_setup(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  int* hdr = WSI(C) + sc.W_HDR; const int ncr = hdr[WH_NCROW], GV = sc.GV;
  if (hdr[WH_RS_NEED] == 0) return;
  int K = 0;
  const bool defer = hdr[WH_RS_DEFER] != 0;   // swept by its own warp in the sweep kernel: its own K
  if (defer) K = hdr[WH_RS_NEED];
  else for (int e2 = C.grp0; e2 < C.grp1; e2++) {
    const int* h2 = (const int*)(as_shared(C.ws) + (long)e2 * sc.w_total) + sc.W_HDR;
    const int k2 = h2[WH_RS_DEFER] ? 0 : h2[WH_RS_NEED]; K = k2 > K ? k2 : K;
  }
  const int nu = hdr[WH_RS_NU], nk = 6 * sc.ncons;
  const RsLayout L = rs_layout(K, nu, nk, ncr / 3);
  if (L.Rp > sc.rs_cap) return;   // (a neighbour's K pads this environment beyond the capacity: dv-space sweeps, WH_RS_R stays 0)
  if (ln == 0) {
    hdr[WH_RS_R] = L.Rp; hdr[WH_RS_K] = K;
#if defined(__CUDA_ARCH__)
    if (C.rs_used) atomicAdd(C.rs_used, 1u);   // how many environment sub-steps needed the row-space solver (steers the schedule)
    if (defer) { const int cls = hdr[WH_RS_DEFER] - 1; const int slot = atomicAdd(C.rs_count + cls, 1); C.rs_lists[(size_t)cls * C.rs_stride + slot] = C.e_local; }
#endif
  }
  float* RSV = WSG(C, sc.X_RSV); float* REC = WSG(C, sc.X_RSREC);
  for (int p = ln; p < L.Rp; p += nt) if (!rs_real(L, p)) { float* rc = REC + RR_W * p; st4(rc, 0.f, 0.f, 0.f, 0.f); st4(rc + 4, 0.f, int_as_float(-1), 0.f, int_as_float(-1)); }
  int r = 0;
  for (int di = 0; di < sc.ndyn; di++) {
    const int* bp = gc(sc.body_plan) + BP_W * gc(sc.dyn_body)[di]; const int n = WSI(C)[sc.W_UCNT + di];
    for (int j = 0; j < n; j++, r++) {
      if (r % nt != ln) continue;
      const float* u = WSH(C, sc.X_UROW) + UR_W * (bp[BP_UROW] + j);
      int col = float_as_int(u[UR_COL]); float sg = 1.f; if (col < 0) { col = -1 - col; sg = -1.f; }
      float* Jd = RSV + (size_t)r * 2 * GV; float* Md = Jd + GV;
      for (int i = 0; i < 2 * GV; i += 4) st4(Jd + i, 0.f, 0.f, 0.f, 0.f);
      const int go = bp[BP_GVOFF], gs = bp[BP_GS]; const float* Mc = WSH(C, sc.W_MINV) + bp[BP_MINVOFF] + col * gs;
      Jd[go + col] = sg;
      for (int i = 0; i < gs; i++) Md[go + i] = sg * Mc[i];
      float* rc = REC + RR_W * r;
      // (RR_APPLIED carries, until the sweeps overwrite it, the support of the row's J: [lo, hi) in floats, lo | hi << 16)
      st4(rc, u[UR_RHS], u[UR_DINV], u[UR_LO], u[UR_HI]); st4(rc + 4, 0.f, int_as_float(-1), int_as_float(((go + col) & ~3) | ((((go + col) & ~3) + 4) << 16)), int_as_float((di << 16) | j));
    }
  }
  // fixed constraints between models (model.py:69-77): three point rows along the world axes, three angular rows
  for (int kr = 0; kr < nk; kr++) {
    const int r2 = L.P1 + kr;
    if (kr % nt != ln) continue;
    const int kc = kr / 6, i = kr % 6;
    const int* ci = gc(sc.cons_i) + DG_CONS_I_W * kc; const float* cf = gc(sc.cons_f) + DG_CONS_F_W * kc;
    const int fa = ci[0], fb = ci[1], ba = body_of_frame(C, fa), bb = body_of_frame(C, fb);
    const float *Ka = KIN(gc(sc.frame_slot)[fa]), *Kb = KIN(gc(sc.frame_slot)[fb]);
    float Pa[3], Pb[3], t[3], err;
    m_vec(t, Ka, cf); v_add(Pa, Ka + 9, t); m_vec(t, Kb, cf + 7); v_add(Pb, Kb + 9, t);
    if (i < 3) err = Pa[i] - Pb[i];
    else {
      float qa[4], qb[4], qaw[4], qbw[4], dq[4];
      mat_to_q(qa, Ka); mat_to_q(qb, Kb); q_mul(qaw, qa, cf + 3); q_mul(qbw, qb, cf + 10);
      const float qbi[4] = {-qbw[0], -qbw[1], -qbw[2], qbw[3]};
      q_mul(dq, qaw, qbi);
      const float vn = v_len(dq); float ang = 2.f * atan2f(vn, dq[3]); if (ang > kPi) ang -= 2.f * kPi;
      err = vn < 1e-12f ? 0.f : dq[i - 3] * ang / vn;
    }
    float e[3] = {0.f, 0.f, 0.f}, ne[3] = {0.f, 0.f, 0.f}; e[i % 3] = 1.f; ne[i % 3] = -1.f;
    float* Jd = RSV + (size_t)r2 * 2 * GV; float* Md = Jd + GV;
    for (int c = 0; c < 2 * GV; c += 4) st4(Jd + c, 0.f, 0.f, 0.f, 0.f);
    float den = 0.f, rel = 0.f, gvl[RS_GVMAX + 8];
    for (int side = 0; side < 2; side++) {
      const int b = side ? bb : ba, f = side ? fb : fa; const int* bp = gc(sc.body_plan) + BP_W * b;
      if (bp[BP_DI] < 0) continue;
      const int go = bp[BP_GVOFF], g = bp[BP_GDIM], gs = bp[BP_GS]; const float* Minv = WSH(C, sc.W_MINV) + bp[BP_MINVOFF];
      if (i < 3) point_jacobian(C, f, side ? Pb : Pa, side ? ne : e, Jd + go); else angular_jacobian(C, f, side ? ne : e, Jd + go);
      body_genvel(C, b, gvl);
      for (int c = 0; c < g; c++) { float sm = 0.f; for (int j = 0; j < g; j++) sm += Minv[j * gs + c] * Jd[go + j]; Md[go + c] = sm; den += Jd[go + c] * sm; rel += Jd[go + c] * gvl[c]; }
    }
    const float dinv = den > 1e-30f ? 1.0f / den : 0.f, lim = cf[14] * sc.dt, hsub = sc.dt / (float)sc.substeps;
    float* rc = REC + RR_W * r2;
    st4(rc, (-rel - err * sc.erp / hsub) * dinv, dinv, -lim, lim); st4(rc + 4, 0.f, int_as_float(-1), int_as_float(0 | (GV << 16)), int_as_float(RS_CONTACT | 0xffff));
  }
  const int nc = ncr / 3;
  for (int rr = 0; rr < ncr; rr++) {
    const int r2 = rr < nc ? L.nrm0 + rr : L.P2 + (rr - nc);
    if (rr % nt != ln) continue;
    const float* row = WSP(C, sc.X_CROW) + sc.crow_stride * rr; const float* J = row + CR_HDR; const float* M = J + sc.GP;
    const int dia = float_as_int(row[CR_DA]), dib = float_as_int(row[CR_DB]);
    float* Jd = RSV + (size_t)r2 * 2 * GV; float* Md = Jd + GV;
    for (int i = 0; i < 2 * GV; i += 4) st4(Jd + i, 0.f, 0.f, 0.f, 0.f);
    int off = 0, slo = GV, shi = 0;
    // (the row was zeroed just above: plain stores, no read-modify-write of global memory, unless both sides are the same body)
    // (loads in batches of four ahead of their stores: the compiler may not move a load of J above a store to Jd - they could
    // alias for all it knows - so a load / store pair per element waits a full memory latency per element)
#define DG_COPY_ROW(dstJ, dstM, srcJ, srcM, g_)                                                                                   \
    { int i_ = 0;                                                                                                                  \
      for (; i_ + 4 <= (g_); i_ += 4) {                                                                                            \
        const float j0_ = (srcJ)[i_], j1_ = (srcJ)[i_ + 1], j2_ = (srcJ)[i_ + 2], j3_ = (srcJ)[i_ + 3];                            \
        const float m0_ = (srcM)[i_], m1_ = (srcM)[i_ + 1], m2_ = (srcM)[i_ + 2], m3_ = (srcM)[i_ + 3];                            \
        (dstJ)[i_] = 0.f + j0_; (dstJ)[i_ + 1] = 0.f + j1_; (dstJ)[i_ + 2] = 0.f + j2_; (dstJ)[i_ + 3] = 0.f + j3_;                \
        (dstM)[i_] = 0.f + m0_; (dstM)[i_ + 1] = 0.f + m1_; (dstM)[i_ + 2] = 0.f + m2_; (dstM)[i_ + 3] = 0.f + m3_;                \
      }                                                                                                                            \
      for (; i_ < (g_); i_++) { const float j0_ = (srcJ)[i_], m0_ = (srcM)[i_]; (dstJ)[i_] = 0.f + j0_; (dstM)[i_] = 0.f + m0_; } }
    if (dia >= 0) { const int* bp = gc(sc.body_plan) + BP_W * gc(sc.dyn_body)[dia]; const int go = bp[BP_GVOFF], g = bp[BP_GDIM]; DG_COPY_ROW(Jd + go, Md + go, J, M, g) off = g; slo = go < slo ? go : slo; shi = go + bp[BP_GS] > shi ? go + bp[BP_GS] : shi; }
    if (dib >= 0) {
      const int* bp = gc(sc.body_plan) + BP_W * gc(sc.dyn_body)[dib]; const int go = bp[BP_GVOFF], g = bp[BP_GDIM];
      if (dib == dia) { for (int i = 0; i < g; i++) { Jd[go + i] += J[off + i]; Md[go + i] += M[off + i]; } }
      else DG_COPY_ROW(Jd + go, Md + go, J + off, M + off, g)
      slo = go < slo ? go : slo; shi = go + bp[BP_GS] > shi ? go + bp[BP_GS] : shi;
    }
    if (shi <= slo) { slo = 0; shi = 0; }
    float* rc = REC + RR_W * r2;
    st4(rc, row[CR_RHS], row[CR_DINV], row[CR_LO], row[CR_HI]); st4(rc + 4, row[CR_MU], row[CR_PARENT], int_as_float(slo | (shi << 16)), int_as_float(RS_CONTACT | rr));
  }
}
#undef DG_COPY_ROW
// A[p * cap + s] = J_s M^-1 J_p^T for real positions p, s < Rp; zero rows / columns for the padding positions and for the
// columns up to K nt that the lanes of the sweeps read
DG_FN void phase_rs_build(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  const RsLayout L = rs_layout_of(C); const int GV = sc.GV, cap = sc.rs_cap;
  int ncol = L.K * nt; if (ncol > cap) ncol = cap; if (ncol < L.Rp) ncol = L.Rp;
  const float* RSV = WSG(C, sc.X_RSV); const float* REC = WSG(C, sc.X_RSREC); float* A = WSG(C, sc.X_RSA);
  // column s of A needs J_s only where it is non-zero: one generalized coordinate for a motor / limit row, the coordinates of the
  // one or two bodies it touches for a contact row (phase_rs_setup left that range in the row record).  The terms left out
  // are exact zeros, so the sums are the ones the full dot products give.
  for (int s2 = ln; s2 < ncol; s2 += nt) {
    const bool rs2 = s2 < L.Rp && rs_real(L, s2);
    int c0 = 0, c1 = 0;
    if (rs2) { const int sup = float_as_int(REC[RR_W * s2 + RR_APPLIED]); c0 = sup & 0xffff; c1 = (sup >> 16) & 0xffff; if (c1 > GV) c1 = GV; }
    const float* Jd = RSV + (size_t)s2 * 2 * GV;
    for (int p = 0; p < L.Rp; p++) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      if (rs2 && rs_real(L, p)) {
        const float* Md = RSV + (size_t)p * 2 * GV + GV;
        for (int c = c0; c < c1; c += 4) { const F4 jv = ld4(Jd + c), mv = ld4(Md + c); a0 = fmaf(jv.x, mv.x, a0); a1 = fmaf(jv.y, mv.y, a1); a2 = fmaf(jv.z, mv.z, a2); a3 = fmaf(jv.w, mv.w, a3); }
      }
      A[p * cap + s2] = (a0 + a1) + (a2 + a3);
    }
  }
}
// dv of every body from the accumulated impulses:  dv = sum_rows (M^-1 J^T)_row x applied_row ; motor / limit impulses back
// into their row records (phase_integrate reports them)
DG_FN void phase_rs_finish(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  const RsLayout L = rs_layout_of(C); const int GV = sc.GV;
  const float* RSV = WSG(C, sc.X_RSV); const float* REC = WSG(C, sc.X_RSREC); float* dv = WSH(C, sc.W_DV);
  for (int i = ln; i < GV; i += nt) {
    float sum = 0.f;
    for (int p = 0; p < L.Rp; p++) if (rs_real(L, p)) sum = fmaf(RSV[(size_t)p * 2 * GV + GV + i], REC[RR_W * p + RR_APPLIED], sum);
    dv[i] = sum;
  }
  for (int r = ln; r < L.nu; r += nt) {
    const int v = float_as_int(REC[RR_W * r + RR_ID]); const int* bp = gc(sc.body_plan) + BP_W * gc(sc.dyn_body)[(v >> 16) & 0x3fff];
    (WSH(C, sc.X_UROW) + UR_W * (bp[BP_UROW] + (v & 0xffff)))[UR_APPLIED] = REC[RR_W * r + RR_APPLIED];
  }
}
#if defined(__CUDA_ARCH__) && defined(DG_STEP_T)
// The sweeps.  Called with the REMAPPED thread layout: the NT lanes of a team are consecutive threads of one warp
// (l = lane in team), every thread of the warp takes part in every shuffle and runs the same sequence of (block, slot)
// steps: the block COUNT of a section is the maximum over the teams of the warp, a team that has fewer blocks idles through
// the surplus steps (no owner, zero broadcast).  FULL: every warp of the block has 32 threads, so the shuffles take the
// literal full mask; a mask held in a register makes nvcc guard every shuffle with MATCH.ANY + REDUX + VOTE.
template <int K> struct RsRow { float v[K]; };
template <int K> __device__ __forceinline__ RsRow<K> rs_ldrow(const float* p) {
  RsRow<K> r;
  if constexpr (K == 2) { const float2 v = *reinterpret_cast<const float2*>(p); r.v[0] = v.x; r.v[1] = v.y; }
  else {
#pragma unroll
    for (int c = 0; c < K / 4; c++) { const float4 v = *reinterpret_cast<const float4*>(p + 4 * c); r.v[4 * c] = v.x; r.v[4 * c + 1] = v.y; r.v[4 * c + 2] = v.z; r.v[4 * c + 3] = v.w; }
  }
  return r;
}
template <int K, int NT, bool FULL>
__device__ __noinline__ void rs_solve_team(const Env& C, const int l, const unsigned wmask_rt, const RsLayout L) {
  const unsigned wmask = FULL ? 0xffffffffu : wmask_rt;
  const DevScene& sc = SC;
  const int tbase = (threadIdx.x & 31) & ~(NT - 1), cap = sc.rs_cap;
  float* REC = WSG(C, sc.X_RSREC); const float* Al = WSG(C, sc.X_RSA) + l * K; float* capp = WSH(C, sc.W_CAPP);
  float rhs[K], dinv[K], lo[K], hi[K], ap[K], y[K], mu[K]; int par[K];
#pragma unroll
  for (int k = 0; k < K; k++) {
    rhs[k] = 0.f; dinv[k] = 0.f; lo[k] = 0.f; hi[k] = 0.f; ap[k] = 0.f; y[k] = 0.f; mu[k] = 0.f; par[k] = -1;
    const int p = l * K + k;
    if (p < L.Rp) { const F4 r0 = ld4(REC + RR_W * p), r1 = ld4(REC + RR_W * p + 4); rhs[k] = r0.x; dinv[k] = r0.y; lo[k] = r0.z; hi[k] = r0.w; mu[k] = r1.x; par[k] = float_as_int(r1.y); }
  }
  // blocks per section of this team, and the step counts of the warp
  const int nb1 = L.P1 / K, nb2 = (L.P2 - L.P1) / K, nb3 = (L.Rp - L.P2) / K, plast = L.Rp > 0 ? L.Rp - 1 : 0;
  const int nb1m = __reduce_max_sync(wmask, nb1), nb2m = __reduce_max_sync(wmask, nb2), nb3m = __reduce_max_sync(wmask, nb3);
  float bprev = 0.f; int pprev = 0;   // broadcast received one step ago and not yet folded into y, and its row
  // one Gauss-Seidel update of position p = jt K + k (jt: block of this team, act: the team has this block).  HAND: first
  // step of a block - the pending broadcast is folded in first, the new owner needs it.  Then every lane evaluates the clamp
  // of ITS slot k; the owner keeps the result, folds its own d into its y at once (the next row's y is its own register) and
  // broadcasts d; the other lanes fold the PREVIOUS broadcast (issued a step ago: no wait).
#define DG_RS_STEP(jt_, act_, k, HAND, NORMAL)                                                                   \
  {                                                                                                              \
    const int jc_ = (jt_) < NT ? (jt_) : NT - 1;                                                                 \
    const int p_ = min(jc_ * K + (k), plast);                                                                    \
    const bool own_ = (act_) && l == (jt_);                                                                      \
    if (HAND) {                                                                                                  \
      const RsRow<K> h_ = rs_ldrow<K>(Al + pprev * cap);                                                         \
      _Pragma("unroll") for (int kk = 0; kk < K; kk++) y[kk] = fmaf(h_.v[kk], bprev, y[kk]);                     \
      bprev = 0.f;                                                                                               \
    }                                                                                                            \
    const RsRow<K> a_ = rs_ldrow<K>(Al + (own_ ? p_ : pprev) * cap);                                             \
    const float new_ = fminf(fmaxf(ap[k] + fmaf(-y[k], dinv[k], rhs[k]), lo[k]), hi[k]);                         \
    const float dl_ = own_ ? new_ - ap[k] : 0.f;                                                                 \
    if (own_) { ap[k] = new_; if ((NORMAL) && p_ >= L.nrm0 && p_ < L.nrm1) capp[p_ - L.nrm0] = new_; }           \
    const float b_ = __shfl_sync(wmask, dl_, tbase + jc_);                                                       \
    const float cf_ = own_ ? dl_ : bprev;                                                                        \
    _Pragma("unroll") for (int kk = 0; kk < K; kk++) y[kk] = fmaf(a_.v[kk], cf_, y[kk]);                         \
    bprev = own_ ? 0.f : b_; pprev = p_;                                                                         \
  }
#define DG_RS_BLOCK_FWD(jt_, act_, NORMAL)                                                                       \
  { _Pragma("unroll") for (int k = 0; k < K; k++) { if (k == 0) DG_RS_STEP(jt_, act_, k, true, NORMAL) else DG_RS_STEP(jt_, act_, k, false, NORMAL) } }
#define DG_RS_BLOCK_REV(jt_, act_)                                                                               \
  { _Pragma("unroll") for (int k = K - 1; k >= 0; k--) { if (k == K - 1) DG_RS_STEP(jt_, act_, k, true, false) else DG_RS_STEP(jt_, act_, k, false, false) } }
  for (int it = 0; it < sc.iters; it++) {
    if (it & 1) { for (int jj = 0; jj < nb1m; jj++) DG_RS_BLOCK_FWD(jj, jj < nb1, false) }
    else { for (int jj = nb1m - 1; jj >= 0; jj--) DG_RS_BLOCK_REV(jj, jj < nb1) }
    for (int jj = 0; jj < nb2m; jj++) DG_RS_BLOCK_FWD(nb1 + jj, jj < nb2, true)
    __syncwarp(wmask);
#pragma unroll
    for (int k = 0; k < K; k++) if (par[k] >= 0) { hi[k] = mu[k] * capp[par[k]]; lo[k] = -hi[k]; }
    for (int jj = 0; jj < nb3m; jj++) DG_RS_BLOCK_FWD(nb1 + nb2 + jj, jj < nb3, false)
  }
#undef DG_RS_BLOCK_FWD
#undef DG_RS_BLOCK_REV
#undef DG_RS_STEP
#pragma unroll
  for (int k = 0; k < K; k++) { const int p = l * K + k; if (p < L.Rp) REC[RR_W * p + RR_APPLIED] = ap[k]; }
}
// remaps the block's threads (thread t -> lane t % NT of the block's environment t / NT) and runs the sweeps
template <int NT>
__device__ __forceinline__ void rs_solve_block(const Env& C) {
  if constexpr (NT >= 2) {
  const DevScene& sc = SC;
  const int E = blockDim.x / NT, ei = threadIdx.x % E, e2 = threadIdx.x / NT, l2 = threadIdx.x % NT;
  Env C2 = C;
  C2.ws = C.ws + (long)(e2 - ei) * sc.w_total; C2.wg = C.wg + (long)(e2 - ei) * sc.g_total;
  const unsigned in_warp = blockDim.x - (threadIdx.x & ~31u);          // threads of this warp that exist
  const unsigned wmask = in_warp >= 32u ? 0xffffffffu : (1u << in_warp) - 1u;
  const int* hdr = WSI(C2) + sc.W_HDR;
  const int R = hdr[WH_RS_DEFER] ? 0 : hdr[WH_RS_R];   // deferred environments are swept by the sweep kernel
  // (R == 0: slot without rows - its other header fields may be stale)
  const RsLayout L = R > 0 ? rs_layout(hdr[WH_RS_K], hdr[WH_RS_NU], 6 * sc.ncons, hdr[WH_NCROW] / 3) : rs_layout(2, 0, 0, 0);
  const int Kw = __reduce_max_sync(wmask, R > 0 ? L.K : 0);   // the same for every environment of the warp that has rows (phase_rs_setup)
  if (Kw > 0) {
    if ((blockDim.x & 31u) == 0u) {
      if (Kw <= 2) rs_solve_team<2, NT, true>(C2, l2, wmask, L);
      else if (Kw <= 4) rs_solve_team<4, NT, true>(C2, l2, wmask, L);
      else rs_solve_team<RS_KMAX, NT, true>(C2, l2, wmask, L);
    } else {
      if (Kw <= 4) rs_solve_team<4, NT, false>(C2, l2, wmask, L);
      else rs_solve_team<RS_KMAX, NT, false>(C2, l2, wmask, L);
    }
  }
  }
}
#elif defined(__CUDA_ARCH__)
template <int NT> __device__ __forceinline__ void rs_solve_block(const Env&) {}
#else
// one-lane form of the same sweeps for the CPU emulation (tests/emul): identical row order and arithmetic
DG_FN void rs_solve_serial(const Env& C, int nt) {
  (void)nt;
  const DevScene& sc = SC;
  const RsLayout L = rs_layout_of(C); const int cap = sc.rs_cap;
  float* REC = WSG(C, sc.X_RSREC); const float* A = WSG(C, sc.X_RSA); float* capp = WSH(C, sc.W_CAPP);
  float lo[RS_KMAX * 32], hi[RS_KMAX * 32], ap[RS_KMAX * 32], y[RS_KMAX * 32];
  for (int p = 0; p < L.Rp; p++) { lo[p] = REC[RR_W * p + RR_LO]; hi[p] = REC[RR_W * p + RR_HI]; ap[p] = 0.f; y[p] = 0.f; }
  auto update = [&](int p, bool normal) {
    const float* rc = REC + RR_W * p;
    const float nw = fminf(fmaxf(ap[p] + fmaf(-y[p], rc[RR_DINV], rc[RR_RHS]), lo[p]), hi[p]), d = nw - ap[p];
    ap[p] = nw;
    if (normal && p >= L.nrm0 && p < L.nrm1) capp[p - L.nrm0] = nw;
    for (int s2 = 0; s2 < L.Rp; s2++) y[s2] = fmaf(A[p * cap + s2], d, y[s2]);
  };
  for (int it = 0; it < sc.iters; it++) {
    if (it & 1) for (int p = 0; p < L.P1; p++) update(p, false); else for (int p = L.P1 - 1; p >= 0; p--) update(p, false);
    for (int p = L.P1; p < L.P2; p++) update(p, true);
    for (int p = L.P2; p < L.fr1; p++) { hi[p] = REC[RR_W * p + RR_MU] * capp[float_as_int(REC[RR_W * p + RR_PAR])]; lo[p] = -hi[p]; }
    for (int p = L.P2; p < L.Rp; p++) update(p, false);
  }
  for (int p = 0; p < L.Rp; p++) REC[RR_W * p + RR_APPLIED] = ap[p];
}
#endif

// ------------------------------------------------------------------ integration --------------------------------
DG_FN void integrate_base_quat(float* q, const float* om, float h) {
  float ang = v_len(om), ax[3];
  if (ang * h > 0.25f * kPi) ang = 0.25f * kPi / h;
  if (ang < 0.001f) v_scale(ax, om, 0.5f * h - h * h * h * 0.020833333333f * ang * ang); else v_scale(ax, om, sinf(0.5f * ang * h) / ang);
  float dq[4] = {ax[0], ax[1], ax[2], cosf(0.5f * ang * h)}, out[4];
  q_mul(out, dq, q); q_norm(out); q[0] = out[0]; q[1] = out[1]; q[2] = out[2]; q[3] = out[3];
}
DG_FN void phase_integrate(const Env& C, int ln, int nt, float h) {
  const DevScene& sc = SC;
  for (int di = ln; di < sc.ndyn; di += nt) {
    int b = gc(sc.dyn_body)[di]; const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int* bp = gc(sc.body_plan) + BP_W * b;
    const float* dv = WSH(C, sc.W_DV) + bp[BP_GVOFF]; int jo = 0;
    // record the motor impulses of this sub-step
    int n = WSI(C)[sc.W_UCNT + di]; const float* rows = WSH(C, sc.X_UROW) + UR_W * bp[BP_UROW];
    for (int j = 0; j < n; j++) { int md = float_as_int(rows[UR_W * j + UR_MOTOR]); if (md >= 0) DOF(D_APPLIED, md) = rows[UR_W * j + UR_APPLIED]; }
    if (bi[0] == 2) {
      float* bs = BST(di);
      for (int i = 0; i < 3; i++) { bs[10 + i] += dv[i]; bs[7 + i] += dv[3 + i]; }
      for (int i = 0; i < 3; i++) bs[i] += h * bs[7 + i];
      integrate_base_quat(bs + 3, bs + 10, h);
      jo = 6;
    }
    for (int i = 0; i < bi[4]; i++) {
      int d = bi[3] + i; float qd = DOF(D_QD, d) + dv[jo + i];
      qd = clampf(qd, -sc.max_joint_vel, sc.max_joint_vel);
      DOF(D_QD, d) = qd; DOF(D_Q, d) += h * qd;
      // SEM_WRENCH_FIRST_SUBSTEP: the applied joint torque leaves the generalized force after the first sub-step (damping stays)
      if ((sc.sem & SEM_WRENCH_FIRST_SUBSTEP) && WSI(C)[sc.W_HDR + WH_SUB] == 0) DOF(D_TAU, d) -= ST(S_JTORQUE)[d];
    }
  }
}
// (after phase_integrate, its own phase: every lane above read the counter)
DG_FN void phase_next_substep(const Env& C, int ln, int nt) { (void)nt; if (ln == 0) WSI(C)[SC.W_HDR + WH_SUB] += 1; }
DG_FN void phase_final_kin(const Env& C, int ln, int nt) {
  for (int di = ln; di < SC.ndyn; di += nt) fk_vel_body<false>(C, gc(SC.dyn_body)[di]);
}
// write the dynamic state back, refresh the link pose / velocity cache the sensors read, clear applied wrenches
DG_FN void phase_store(const Env& C, int ln, int nt, int clear_forces) {
  const DevScene& sc = SC;
  for (int i = ln; i < 13 * sc.ndyn; i += nt) {
    int di = i / 13, k = i - 13 * di, b = gc(sc.dyn_body)[di]; float v = BST(di)[k];
    if (k < 3) ST(S_BPOS)[3 * b + k] = v;
    else if (k < 7) ST(S_BQUAT)[4 * b + k - 3] = v;
    else if (k < 10) ST(S_BVEL)[3 * b + k - 7] = v;
    else ST(S_BOMEGA)[3 * b + k - 10] = v;
  }
  for (int d = ln; d < sc.nd; d += nt) {
    ST(S_Q)[d] = DOF(D_Q, d); ST(S_QD)[d] = DOF(D_QD, d); ST(S_MAPPLIED)[d] = DOF(D_APPLIED, d);
    if (clear_forces) ST(S_JTORQUE)[d] = 0.f;
  }
  for (int gl = ln; gl < sc.nl; gl += nt) {
    int s = gc(sc.frame_slot)[sc.nb + gl];
    if (s < 0) continue;
    const float* K = KIN(s); float q[4], t[3];
    v_cpy(ST(S_LPOS) + 3 * gl, K + 9);
    mat_to_q(q, K); for (int i = 0; i < 4; i++) ST(S_LQUAT)[4 * gl + i] = q[i];
    const float* V = ABA(s) + AB_WV;
    m_vec(t, K, V + 3); v_cpy(ST(S_LVEL) + 3 * gl, t);
    m_vec(t, K, V); v_cpy(ST(S_LOMEGA) + 3 * gl, t);
  }
  if (clear_forces) for (int f = ln; f < sc.nframes; f += nt) {
    if (gc(sc.frame_slot)[f] < 0) continue;
    for (int i = 0; i < 3; i++) { ST(S_EXTF)[3 * f + i] = 0.f; ST(S_EXTT)[3 * f + i] = 0.f; }
  }
}

// ------------------------------------------------------------------ frame queries on the state row -------------
// COM-frame pose and velocity as cached after the last step (what the reference reads through
// getBasePositionAndOrientation / getLinkState[0,1,6,7], e.g. object_state_sensor.py:33-48)
DG_FN void frame_com_state(const Env& C, int f, float* pos, float* quat, float* vel, float* om) {
  const DevScene& sc = SC;
  if (f < sc.nb) { v_cpy(pos, ST(S_BPOS) + 3 * f); for (int i = 0; i < 4; i++) quat[i] = ST(S_BQUAT)[4 * f + i]; v_cpy(vel, ST(S_BVEL) + 3 * f); v_cpy(om, ST(S_BOMEGA) + 3 * f); }
  else { int gl = f - sc.nb; v_cpy(pos, ST(S_LPOS) + 3 * gl); for (int i = 0; i < 4; i++) quat[i] = ST(S_LQUAT)[4 * gl + i]; v_cpy(vel, ST(S_LVEL) + 3 * gl); v_cpy(om, ST(S_LOMEGA) + 3 * gl); }
}
// URDF link-frame pose (getLinkState[4,5]; reach_target.py:21-30, camera.py:60)
DG_FN void frame_link_pose(const Env& C, int f, float* pos, float* quat) {
  float v[3], o[3];
  frame_com_state(C, f, pos, quat, v, o);
  if (f >= SC.nb) {
    const float* lf = C.link_f + DG_LINK_F_W * (f - SC.nb);
    float R[9], t[3], qi[4] = {-lf[16], -lf[17], -lf[18], lf[19]}, qo[4];
    q_to_mat(R, quat); m_vec(t, R, lf + 7); v_sub(pos, pos, t);
    q_mul(qo, quat, qi); for (int i = 0; i < 4; i++) quat[i] = qo[i];
  }
}

// ------------------------------------------------------------------ inverse kinematics -------------------------
// In-place Gaussian elimination with partial pivoting on workspace arrays
DG_FN int solve_dense(float* A, float* bvec, int n) {
  for (int c = 0; c < n; c++) {
    int p = c;
    for (int r2 = c + 1; r2 < n; r2++) if (fabsf(A[r2 * n + c]) > fabsf(A[p * n + c])) p = r2;
    if (fabsf(A[p * n + c]) < 1e-30f) return -1;
    if (p != c) { for (int j = 0; j < n; j++) { float t = A[c * n + j]; A[c * n + j] = A[p * n + j]; A[p * n + j] = t; } float t = bvec[c]; bvec[c] = bvec[p]; bvec[p] = t; }
    for (int r2 = c + 1; r2 < n; r2++) { float f = A[r2 * n + c] / A[c * n + c]; if (f != 0.f) { for (int j = c; j < n; j++) A[r2 * n + j] -= f * A[c * n + j]; bvec[r2] -= f * bvec[c]; } }
  }
  for (int r2 = n - 1; r2 >= 0; r2--) { float s = bvec[r2]; for (int j = r2 + 1; j < n; j++) s -= A[r2 * n + j] * bvec[j]; bvec[r2] = s / A[r2 * n + r2]; }
  return 0;
}
// Damped least squares on the end-effector link frame in base coordinates over all DoF of body b
// (what ik_controller.py:61-69 asks of calculateInverseKinematics); result in scr[0 .. nd_b)
DG_FN void ik_solve(const Env& C, int b, int ee_gl, const float* tpos_w, const float* torn_w, int use_orn, int nullspace,
                    const float* lower, const float* upper, const float* range, const float* rest, float* scr) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; int d0 = bi[3], ndb = bi[4];
  int mc = sc.max_depth + 2;
  float* qb = scr; float* nullv = qb + ndb; float* dth = nullv + ndb; float* J = dth + ndb;     // J: 6 x ndb
  float* A = J + 6 * ndb; int asz = ndb * ndb > 36 ? ndb * ndb : 36;
  float* rhs = A + asz; float* axw = rhs + (ndb > 6 ? ndb : 6); float* orgw = axw + 3 * mc;
  int* chain = (int*)(orgw + 3 * mc);
  for (int i = 0; i < ndb; i++) qb[i] = ST(S_Q)[d0 + i];
  const float *bp = ST(S_BPOS) + 3 * b, *bq = ST(S_BQUAT) + 4 * b;
  float Rb[9], tp[3], d[3], tq[4] = {0, 0, 0, 1};
  q_to_mat(Rb, bq); v_sub(d, tpos_w, bp); mT_vec(tp, Rb, d);
  if (use_orn) { float bqi[4] = {-bq[0], -bq[1], -bq[2], bq[3]}; q_mul(tq, bqi, torn_w); }
  if (nullspace) for (int i = 0; i < ndb; i++) {
    float nv = 0.001f * (rest[i] - qb[i]);
    if (qb[i] > upper[i]) nv += 10.0f * (upper[i] - qb[i]) / range[i];
    if (qb[i] < lower[i]) nv += 10.0f * (lower[i] - qb[i]) / range[i];
    nullv[i] = nv;
  }
  int nc = 0;
  for (int gl = ee_gl; gl >= 0; gl = shc(C.link_i)[DG_LINK_I_W * gl + 1]) chain[nc++] = gl;
  int m = use_orn ? 6 : 3;
  float diff = 1e30f;
  for (int it = 0; it < sc.ik_iters && diff > sc.ik_threshold; it++) {
    // forward kinematics of the chain in base coordinates + geometric Jacobian
    float Rc[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, pc[3] = {0, 0, 0};
    for (int i = nc - 1; i >= 0; i--) {
      int gl = chain[i]; const int* li = shc(C.link_i) + DG_LINK_I_W * gl; const float* lf = shc(C.link_f) + DG_LINK_F_W * gl;
      float E[9], r[3], t[3], Rn[9];
      joint_xform(C, gl, li[3] >= 0 ? qb[li[3] - d0] : 0.0f, E, r);
      m_vec(t, Rc, r); v_add(pc, pc, t); m_mulT(Rn, Rc, E); m_cpy(Rc, Rn);
      m_vec(axw + 3 * i, Rc, lf + 10);
      float dw[3]; m_vec(dw, Rc, lf + 7); v_sub(orgw + 3 * i, pc, dw);
    }
    const float* lfe = shc(C.link_f) + DG_LINK_F_W * ee_gl;
    float pos[3], R[9], dw[3], Rli[9], qi[4] = {-lfe[16], -lfe[17], -lfe[18], lfe[19]};
    m_vec(dw, Rc, lfe + 7); v_sub(pos, pc, dw);
    q_to_mat(Rli, qi); m_mul(R, Rc, Rli);
    for (int i = 0; i < 6 * ndb; i++) J[i] = 0.f;
    for (int i = 0; i < nc; i++) {
      const int* li = shc(C.link_i) + DG_LINK_I_W * chain[i];
      if (li[3] < 0) continue;
      int jd = li[3] - d0;
      if (li[2] == 1) { float rel[3], t[3]; v_sub(rel, pos, orgw + 3 * i); v_cross(t, axw + 3 * i, rel); for (int k = 0; k < 3; k++) { J[k * ndb + jd] = t[k]; J[(3 + k) * ndb + jd] = axw[3 * i + k]; } }
      else if (li[2] == 2) for (int k = 0; k < 3; k++) J[k * ndb + jd] = axw[3 * i + k];
    }
    float e[6];
    v_sub(e, tp, pos); diff = v_len(e);
    if (use_orn) {
      float qc[4], qci[4], dq[4]; mat_to_q(qc, R); qci[0] = -qc[0]; qci[1] = -qc[1]; qci[2] = -qc[2]; qci[3] = qc[3];
      q_mul(dq, tq, qci);
      // axis * angle of dq; same value as 2 acos(w) with axis xyz / sqrt(1 - w^2), written with atan2 on |xyz|
      // because acos loses half the fp32 mantissa for the small rotations this controller asks for
      float vn = v_len(dq), ax[3];
      float ang = 2 * atan2f(vn, dq[3]);
      if (vn * vn < 10 * 2.220446049250313e-16f) v_set(ax, 1, 0, 0); else v_scale(ax, dq, 1.0f / vn);
      if (ang > kPi) ang -= 2 * kPi; else if (ang < -kPi) ang += 2 * kPi;
      v_scale(e + 3, ax, ang);
    }
    if (!nullspace) {   // dth = (J^T J + lam I)^-1 J^T e
      for (int i = 0; i < ndb; i++) {
        for (int j = 0; j < ndb; j++) { float s = 0.f; for (int k = 0; k < m; k++) s += J[k * ndb + i] * J[k * ndb + j]; A[i * ndb + j] = s + (i == j ? sc.ik_damping : 0.f); }
        float s = 0.f; for (int k = 0; k < m; k++) s += J[k * ndb + i] * e[k]; rhs[i] = s;
      }
      if (solve_dense(A, rhs, ndb) != 0) break;
      for (int i = 0; i < ndb; i++) dth[i] = rhs[i];
    } else {            // dth = J^T (J J^T + lam2 I)^-1 (e - J n) + n
      for (int i = 0; i < m; i++) { float s = 0.f; for (int k = 0; k < ndb; k++) s += J[i * ndb + k] * nullv[k]; rhs[i] = e[i] - s; }
      for (int i = 0; i < m; i++) for (int j = 0; j < m; j++) { float s = 0.f; for (int k = 0; k < ndb; k++) s += J[i * ndb + k] * J[j * ndb + k]; A[i * m + j] = s + (i == j ? sc.ik_null_lambda_sq : 0.f); }
      if (solve_dense(A, rhs, m) != 0) break;
      for (int k = 0; k < ndb; k++) { float s = nullv[k]; for (int i = 0; i < m; i++) s += J[i * ndb + k] * rhs[i]; dth[k] = s; }
    }
    float mx = 0.f; for (int i = 0; i < ndb; i++) mx = fmaxf(mx, fabsf(dth[i]));
    float cap = 45.0f * kPi / 180.0f;
    if (mx > cap) for (int i = 0; i < ndb; i++) dth[i] *= cap / mx;
    for (int i = 0; i < ndb; i++) qb[i] += dth[i];
  }
}

// Register-resident form of ik_solve for bodies with at most MAXD DoF and M = 3 (position) or 6 (pose) task rows.
// Both damping variants reduce to  dth = J^T (J J^T + lam I)^-1 (e - J n) + n  (n = 0 without null-space terms, by
// the push-through identity (J^T J + lam I)^-1 J^T = J^T (J J^T + lam I)^-1), so only an M x M SPD system is solved.
template <int MAXD, int M>
DG_FN void ik_solve_fast(const Env& C, int b, int ee_gl, const float* tpos_w, const float* torn_w, int nullspace,
                         const float* lower, const float* upper, const float* range, const float* rest, float* scr) {
  const DevScene& sc = SC;
  const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int d0 = bi[3], ndb = bi[4];
  const int mc = sc.max_depth + 2;
  float* qb = scr; float* axw = scr + MAXD; float* orgw = axw + 3 * mc;
  int* chain = (int*)(orgw + 3 * mc); int* cpos = chain + mc;
  float nullv[MAXD];
#pragma unroll
  for (int k = 0; k < MAXD; k++) { nullv[k] = 0.f; if (k < ndb) { qb[k] = ST(S_Q)[d0 + k]; cpos[k] = -1; } }
  const float *bp = ST(S_BPOS) + 3 * b, *bq = ST(S_BQUAT) + 4 * b;
  float Rb[9], tp[3], d[3], tq[4] = {0, 0, 0, 1};
  q_to_mat(Rb, bq); v_sub(d, tpos_w, bp); mT_vec(tp, Rb, d);
  if (M == 6) { float bqi[4] = {-bq[0], -bq[1], -bq[2], bq[3]}; q_mul(tq, bqi, torn_w); }
  if (nullspace) {
#pragma unroll
    for (int k = 0; k < MAXD; k++) if (k < ndb) {
      float q = qb[k], nv = 0.001f * (rest[k] - q);
      if (q > upper[k]) nv += 10.0f * (upper[k] - q) / range[k];
      if (q < lower[k]) nv += 10.0f * (lower[k] - q) / range[k];
      nullv[k] = nv;
    }
  }
  int nc = 0;
  for (int gl = ee_gl; gl >= 0; gl = shc(C.link_i)[DG_LINK_I_W * gl + 1]) { int dof = shc(C.link_i)[DG_LINK_I_W * gl + 3]; if (dof >= 0) cpos[dof - d0] = nc; chain[nc++] = gl; }
  const float lam = nullspace ? sc.ik_null_lambda_sq : sc.ik_damping;
  const float* lfe = shc(C.link_f) + DG_LINK_F_W * ee_gl;
  float Rli[9]; { float qi[4] = {-lfe[16], -lfe[17], -lfe[18], lfe[19]}; q_to_mat(Rli, qi); }
  float diff = 1e30f;
  for (int it = 0; it < sc.ik_iters && diff > sc.ik_threshold; it++) {
    float Rc[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, pc[3] = {0, 0, 0};
    for (int i = nc - 1; i >= 0; i--) {
      int gl = chain[i]; const int* li = shc(C.link_i) + DG_LINK_I_W * gl; const float* lf = shc(C.link_f) + DG_LINK_F_W * gl;
      float E[9], r[3], t[3], Rn[9];
      joint_xform(C, gl, li[3] >= 0 ? qb[li[3] - d0] : 0.0f, E, r);
      m_vec(t, Rc, r); v_add(pc, pc, t); m_mulT(Rn, Rc, E); m_cpy(Rc, Rn);
      if (li[3] >= 0) { m_vec(axw + 3 * i, Rc, lf + 10); float dw[3]; m_vec(dw, Rc, lf + 7); v_sub(orgw + 3 * i, pc, dw); }
    }
    float pos[3], dw[3];
    m_vec(dw, Rc, lfe + 7); v_sub(pos, pc, dw);
    float J[M][MAXD];
#pragma unroll
    for (int k = 0; k < MAXD; k++) {
#pragma unroll
      for (int r = 0; r < M; r++) J[r][k] = 0.f;
      if (k < ndb && cpos[k] >= 0) {
        int i = cpos[k]; const float* ax = axw + 3 * i;
        if (shc(C.link_i)[DG_LINK_I_W * chain[i] + 2] == 1) {
          float rel[3], t[3]; v_sub(rel, pos, orgw + 3 * i); v_cross(t, ax, rel);
          J[0][k] = t[0]; J[1][k] = t[1]; J[2][k] = t[2];
          if (M == 6) { J[M - 3][k] = ax[0]; J[M - 2][k] = ax[1]; J[M - 1][k] = ax[2]; }
        } else { J[0][k] = ax[0]; J[1][k] = ax[1]; J[2][k] = ax[2]; }
      }
    }
    float e[M];
    { float e3[3]; v_sub(e3, tp, pos); diff = v_len(e3); e[0] = e3[0]; e[1] = e3[1]; e[2] = e3[2]; }
    if (M == 6) {
      float R[9], qc[4], qci[4], dq[4]; m_mul(R, Rc, Rli); mat_to_q(qc, R); qci[0] = -qc[0]; qci[1] = -qc[1]; qci[2] = -qc[2]; qci[3] = qc[3];
      q_mul(dq, tq, qci);
      float vn = v_len(dq), ax[3];
      float ang = 2 * atan2f(vn, dq[3]);
      if (vn * vn < 10 * 2.220446049250313e-16f) v_set(ax, 1, 0, 0); else v_scale(ax, dq, 1.0f / vn);
      if (ang > kPi) ang -= 2 * kPi; else if (ang < -kPi) ang += 2 * kPi;
      e[M - 3] = ax[0] * ang; e[M - 2] = ax[1] * ang; e[M - 1] = ax[2] * ang;
    }
    // y = e - J n ;  U = J J^T + lam I (lower triangle) ; solve U x = y by LDL^T without pivoting (U is SPD)
    float x[M], U[M][M];
#pragma unroll
    for (int r = 0; r < M; r++) {
      float sdot = 0.f;
#pragma unroll
      for (int k = 0; k < MAXD; k++) sdot = fmaf(J[r][k], nullv[k], sdot);
      x[r] = e[r] - sdot;
#pragma unroll
      for (int c = 0; c <= r; c++) {
        float u = 0.f;
#pragma unroll
        for (int k = 0; k < MAXD; k++) u = fmaf(J[r][k], J[c][k], u);
        U[r][c] = u + (r == c ? lam : 0.f);
      }
    }
#pragma unroll
    for (int c = 0; c < M; c++) {            // forward elimination on the lower triangle (columns below the pivot)
      float inv = 1.0f / U[c][c];
#pragma unroll
      for (int r = c + 1; r < M; r++) {
        float urc = U[r][c], f = urc * inv;
#pragma unroll
        for (int c2 = c + 1; c2 < r; c2++) U[r][c2] -= urc * U[c2][c];   // U[c2][c] already holds L[c2][c]
        U[r][r] -= urc * f;
        x[r] -= f * x[c];
        U[r][c] = f;                          // keep L for the back substitution
      }
    }
#pragma unroll
    for (int r = M - 1; r >= 0; r--) {        // back substitution with U^T = D L^T
      float sdot = x[r] / U[r][r];
#pragma unroll
      for (int r2 = r + 1; r2 < M; r2++) sdot -= U[r2][r] * x[r2];
      x[r] = sdot;
    }
    float dth[MAXD], mx = 0.f;
#pragma unroll
    for (int k = 0; k < MAXD; k++) {
      float sdot = nullv[k];
#pragma unroll
      for (int r = 0; r < M; r++) sdot = fmaf(J[r][k], x[r], sdot);
      dth[k] = sdot; mx = fmaxf(mx, fabsf(sdot));
    }
    const float cap = 45.0f * kPi / 180.0f;
    float sc_ = mx > cap ? cap / mx : 1.0f;
#pragma unroll
    for (int k = 0; k < MAXD; k++) if (k < ndb) qb[k] += dth[k] * sc_;
  }
}
DG_FN void ik_solve_any(const Env& C, int b, int ee_gl, const float* tpos_w, const float* torn_w, int use_orn, int nullspace,
                        const float* lower, const float* upper, const float* range, const float* rest, float* scr) {
  const int ndb = gc(SC.body_i)[DG_BODY_I_W * b + 4];
  if (ndb <= 6) { if (use_orn) ik_solve_fast<6, 6>(C, b, ee_gl, tpos_w, torn_w, nullspace, lower, upper, range, rest, scr); else ik_solve_fast<6, 3>(C, b, ee_gl, tpos_w, torn_w, nullspace, lower, upper, range, rest, scr); }
  else if (ndb <= 12) { if (use_orn) ik_solve_fast<12, 6>(C, b, ee_gl, tpos_w, torn_w, nullspace, lower, upper, range, rest, scr); else ik_solve_fast<12, 3>(C, b, ee_gl, tpos_w, torn_w, nullspace, lower, upper, range, rest, scr); }
  else ik_solve(C, b, ee_gl, tpos_w, torn_w, use_orn, nullspace, lower, upper, range, rest, scr);
}

// ------------------------------------------------------------------ add-on ops ---------------------------------
DG_FN void admittance_update(const Env& C, const int* ia, const float* fa, const float* a);
// controllers: update() bodies of /root/reference/diy_gym/addons/controllers/
DG_FN void phase_actions(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  int ik_seen = 0;
  for (int k = 0; k < sc.nop; k++) {
    const int* op = gc(sc.op_i) + DG_OP_I_W * k; const int* ia = gc(sc.oparg_i) + op[1]; const float* fa = gc(sc.oparg_f) + op[2];
    const float* a = op[3] >= 0 ? C.act + op[3] : nullptr;
    if (k < 128 && !((C.opmask[k >> 6] >> (k & 63)) & 1ull)) { if (op[0] == OP_IK_CTRL) ik_seen++; continue; }
    if (op[0] == OP_JOINT_CTRL && ln == 0) {                 // joint_controller.py:40-58
      int mode = ia[0], n = ia[1];
      for (int i = 0; i < n; i++) {
        int d = ia[2 + i];
        if (mode == 2) { ST(S_JTORQUE)[d] += a[i]; continue; }
        ST(S_MKD)[d] = fa[1]; ST(S_MMAXF)[d] = fa[2 + i];
        if (mode == 0) { ST(S_MKP)[d] = fa[0]; ST(S_MTPOS)[d] = a[i]; ST(S_MTVEL)[d] = 0.f; }
        else { ST(S_MKP)[d] = 0.f; ST(S_MTPOS)[d] = 0.f; ST(S_MTVEL)[d] = a[i]; }
      }
    } else if (op[0] == OP_EXT_FORCE && ln == 0) {           // external_force.py:21-24 (+ LINK_FRAME variant, drone_pilot.py:35-37)
      int f = ia[0]; float pos[3], quat[4], v[3], o[3], F[3], rel[3], t[3];
      frame_com_state(C, f, pos, quat, v, o);
      if (ia[1] == 0) { v_cpy(F, a); v_sub(rel, fa, pos); }
      else { float R[9]; q_to_mat(R, quat); m_vec(F, R, a); m_vec(rel, R, fa); }
      v_add(ST(S_EXTF) + 3 * f, ST(S_EXTF) + 3 * f, F); v_cross(t, rel, F); v_add(ST(S_EXTT) + 3 * f, ST(S_EXTT) + 3 * f, t);
    } else if (op[0] == OP_FILTERED_WRENCH && ln == 0) {     // user add-ons lowered to the kernel: examples/drone_pilot Propellor
      // (drone_pilot.py:31-37 of the reference): first-order filter of the action, link-frame force / torque scaled by its state
      float* st_ = ST(S_ADDON) + ia[2]; const float s_ = st_[0] + (a[0] - st_[0]) * fa[0];
      st_[0] = s_;
      const int f = ia[0]; float pos[3], quat[4], v[3], o[3], R[9], F[3], T[3], rel[3], t[3];
      frame_com_state(C, f, pos, quat, v, o); q_to_mat(R, quat);
      const float Fl[3] = {fa[1] * s_, fa[2] * s_, fa[3] * s_}, Tl[3] = {fa[4] * s_, fa[5] * s_, fa[6] * s_};
      m_vec(F, R, Fl); m_vec(T, R, Tl); m_vec(rel, R, fa + 7);
      v_add(ST(S_EXTF) + 3 * f, ST(S_EXTF) + 3 * f, F); v_cross(t, rel, F); v_add(t, t, T); v_add(ST(S_EXTT) + 3 * f, ST(S_EXTT) + 3 * f, t);
    } else if (op[0] == OP_ADMITTANCE && ln == 0) {          // admittance_controller.py:36-55
      admittance_update(C, ia, fa, a);
    } else if (op[0] == OP_IK_CTRL) {                         // ik_controller.py:51-80
      int mine = (ik_seen++ % nt) == ln;
      if (!mine) continue;
      int b = ia[0], ee = ia[1], n = ia[2], use_orn = ia[3], nsp = ia[4]; int ndb = gc(sc.body_i)[DG_BODY_I_W * b + 4];
      float pos[3], quat[4], v[3], o[3], tq[4] = {0, 0, 0, 1};
      frame_com_state(C, sc.nb + ee, pos, quat, v, o);
      float tpos[3] = {pos[0] + a[0], pos[1] + a[1], pos[2] + a[2]};
      if (use_orn) { float dq[4]; q_from_euler(dq, a + 3); q_mul(tq, quat, dq); }
      const float* lim = fa + 2 + n;
      float* scr = WSG(C, sc.X_IK) + sc.ik_stride * (ln % (sc.n_ik < nt ? sc.n_ik : nt));
      ik_solve_any(C, b, ee, tpos, tq, use_orn, nsp, lim, lim + ndb, lim + 2 * ndb, lim + 3 * ndb, scr);
      for (int i = 0; i < n; i++) {
        int d = ia[5 + i];
        ST(S_MKP)[d] = fa[0]; ST(S_MKD)[d] = fa[1]; ST(S_MMAXF)[d] = fa[2 + i]; ST(S_MTPOS)[d] = scr[i]; ST(S_MTVEL)[d] = 0.f;
      }
    }
  }
  if (ln == 0) ST(S_STEP)[0] += 1.f;
}
// world-space axis and origin of the joint that carries link gl, from the cached link poses (same construction as point_jacobian)
DG_FN void joint_axis_world(const Env& C, int gl, float* aw, float* ow) {
  const float* lf = shc(C.link_f) + DG_LINK_F_W * gl;
  float R[9], dw[3];
  q_to_mat(R, ST(S_LQUAT) + 4 * gl); m_vec(aw, R, lf + 10); m_vec(dw, R, lf + 7); v_sub(ow, ST(S_LPOS) + 3 * gl, dw);
}
// admittance_controller.py:36-55: tau = F . J_lin + T . J_ang (Jacobian of the admittance point, p.calculateJacobian)
//   + gravity torques (p.calculateInverseDynamics at zero velocity / acceleration) + kp (target - q) - kd qd, applied as
// joint torques (TORQUE_CONTROL).  Fixed-base bodies; the joint list spans every DoF of the body (the host layer checks).
DG_FN void admittance_update(const Env& C, const int* ia, const float* fa, const float* a) {
  const DevScene& sc = SC;
  const int b = ia[0], ee = ia[1], n = ia[2]; const int* bi = gc(sc.body_i) + DG_BODY_I_W * b; const int l0 = bi[1], nlb = bi[2];
  const float kp = fa[0], kd = fa[1]; const float* target = fa + 5;
  for (int i = 0; i < n; i++) { const int d = ia[3 + i]; ST(S_JTORQUE)[d] += (target[i] - ST(S_Q)[d]) * kp - kd * ST(S_QD)[d]; }
  float Re[9], P[3], t[3];
  q_to_mat(Re, ST(S_LQUAT) + 4 * ee); m_vec(t, Re, fa + 2); v_add(P, ST(S_LPOS) + 3 * ee, t);   // admittance point (offset in the link's COM frame)
  for (int gl = ee; gl >= 0; gl = shc(C.link_i)[DG_LINK_I_W * gl + 1]) {
    const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
    if (li[3] < 0) continue;
    float aw[3], ow[3], rel[3], c[3];
    joint_axis_world(C, gl, aw, ow);
    if (li[2] == 1) { v_sub(rel, P, ow); v_cross(c, aw, rel); ST(S_JTORQUE)[li[3]] += v_dot(a, c) + v_dot(a + 3, aw); }
    else ST(S_JTORQUE)[li[3]] += v_dot(a, aw);
  }
  for (int k = 0; k < nlb; k++) {   // G(q): every link's weight through the joints above it
    const float m = PR(P_MASS)[sc.nb + l0 + k];
    if (m == 0.f) continue;
    const float* pk = ST(S_LPOS) + 3 * (l0 + k);
    for (int gl = l0 + k; gl >= 0; gl = shc(C.link_i)[DG_LINK_I_W * gl + 1]) {
      const int* li = shc(C.link_i) + DG_LINK_I_W * gl;
      if (li[3] < 0) continue;
      float aw[3], ow[3], rel[3], c[3];
      joint_axis_world(C, gl, aw, ow);
      if (li[2] == 1) { v_sub(rel, pk, ow); v_cross(c, aw, rel); } else v_cpy(c, aw);
      ST(S_JTORQUE)[li[3]] -= m * v_dot(sc.g, c);
    }
  }
}
// sensors / rewards / terminals: observe(), reward(), is_terminal() bodies of diy_gym/addons/{sensors,rewards}/
DG_FN void phase_observe(const Env& C, int ln, int nt) {
  const DevScene& sc = SC;
  for (int k = ln; k < sc.nop; k += nt) {
    const int* op = gc(sc.op_i) + DG_OP_I_W * k; const int* ia = gc(sc.oparg_i) + op[1]; const float* fa = gc(sc.oparg_f) + op[2];
    float* o = op[4] >= 0 ? C.obs + op[4] : nullptr;
    if (op[0] == OP_JOINT_SENSOR) {                     // joint_state_sensor.py:46-57
      int n = ia[0], flags = ia[1], j = 0;
      for (int i = 0; i < n; i++) o[j++] = ST(S_Q)[ia[2 + i]];
      if (flags & 1) for (int i = 0; i < n; i++) o[j++] = ST(S_QD)[ia[2 + i]];
      if (flags & 2) for (int i = 0; i < n; i++) o[j++] = ST(S_MAPPLIED)[ia[2 + i]] / sc.dt;
    } else if (op[0] == OP_OBJECT_SENSOR) {             // object_state_sensor.py:33-75
      float p[3], q[4], v[3], w[3]; int flags = ia[2], j = 0;
      frame_com_state(C, ia[0], p, q, v, w);
      if (ia[1] >= 0) {
        float sp[3], sq[4], sv[3], sw[3], qq[4];
        frame_com_state(C, ia[1], sp, sq, sv, sw);
        v_sub(p, p, sp); v_sub(v, v, sv); q_mul(qq, sq, q); for (int i = 0; i < 4; i++) q[i] = qq[i]; v_sub(w, w, sw);
      }
      for (int i = 0; i < 3; i++) o[j++] = p[i];
      if (flags & 2) for (int i = 0; i < 3; i++) o[j++] = v[i];
      if (flags & 1) { float e[3]; euler_from_q(e, q); for (int i = 0; i < 3; i++) o[j++] = e[i]; }
      if ((flags & 3) == 3) for (int i = 0; i < 3; i++) o[j++] = w[i];
    } else if (op[0] == OP_FT_SENSOR) {                 // force_torque_sensor.py:21-23
      for (int i = 0; i < 6; i++) o[i] = ST(S_JREACT)[6 * ia[0] + i];
    } else if (op[0] == OP_REACH_TARGET) {              // reach_target.py:21-36
      float sp[3], sq[4], tp[3], tq[4], d[3];
      frame_link_pose(C, ia[0], sp, sq); frame_link_pose(C, ia[1], tp, tq); v_sub(d, tp, sp);
      float dist = v_len(d);
      C.rew[op[5]] = -dist * fa[0]; C.term[op[6]] = dist < fa[1];
    } else if (op[0] == OP_ELECTRICITY) {               // electricity_cost.py:15-18
      const int* bi = gc(sc.body_i) + DG_BODY_I_W * ia[0]; float s = 0.f;
      for (int i = 0; i < bi[4]; i++) s += fabsf(ST(S_MAPPLIED)[bi[3] + i] / sc.dt * ST(S_QD)[bi[3] + i]);
      C.rew[op[5]] = -s * fa[0];
    } else if (op[0] == OP_STUCK_JOINT) {               // stuck_joint_cost.py:19-21 (intent; the reference raises NameError)
      const int* bi = gc(sc.body_i) + DG_BODY_I_W * ia[0]; int stuck = 0;
      for (int l = 0; l < bi[2]; l++) {
        const int* li = shc(C.link_i) + DG_LINK_I_W * (bi[1] + l); const float* lf = shc(C.link_f) + DG_LINK_F_W * (bi[1] + l);
        if (li[3] < 0) continue;
        float qq = ST(S_Q)[li[3]];
        if (fminf(fabsf(lf[20] - qq), fabsf(lf[21] - qq)) < 0.01f) stuck = 1;
      }
      C.rew[op[5]] = stuck ? -fa[0] : 0.0f;
    } else if (op[0] == OP_TIME_PENALTY) {              // time_penalty.py:11-12
      C.rew[op[5]] = fa[0];
    } else if (op[0] == OP_FILTERED_WRENCH) {           // Propellor.observe: the filter state (drone_pilot.py:39-40)
      o[0] = ST(S_ADDON)[ia[2]];
    } else if (op[0] == OP_TILT_TERMINAL) {             // FellOver.is_terminal (drone_pilot.py:52-55): base tilted by more than fa[0] rad
      const float* q = ST(S_BQUAT) + 4 * ia[0];
      C.term[op[6]] = 2.0f * atan2f(sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2]), fabsf(q[3])) > fa[0];
    } else if (op[0] == OP_EPISODE_TIMER) {             // diy_gym.py:180-183
      C.term[op[6]] = ST(S_STEP)[0] >= fa[0];
    }
  }
}
// reset() bodies of joint/ik controllers, respawn, dynamics_randomizer (diy_gym.py:139-143)
DG_FN void phase_reset_ops(const Env& C, int ln, int nt) {
  if (ln != 0) return;
  const DevScene& sc = SC;
  ST(S_STEP)[0] = 0.f;
  uint32_t epoch = (uint32_t)ST(S_RESETS)[0];
  for (int k = 0; k < sc.nop; k++) {
    const int* op = gc(sc.op_i) + DG_OP_I_W * k; const int* ia = gc(sc.oparg_i) + op[1]; const float* fa = gc(sc.oparg_f) + op[2];
    if (op[0] == OP_FILTERED_WRENCH) {                  // ia[1]: clear the filter state on reset (the reference's Propellor keeps it)
      if (ia[1]) ST(S_ADDON)[ia[2]] = 0.f;
    } else if (op[0] == OP_JOINT_RESET) {               // joint_controller.py:36-38, ik_controller.py:47-49
      for (int i = 0; i < ia[0]; i++) { ST(S_Q)[ia[1 + i]] = fa[i]; ST(S_QD)[ia[1 + i]] = 0.f; }
    } else if (op[0] == OP_RESPAWN) {                   // respawn.py:31-39
      int b = ia[0]; uint32_t ep = ia[1] ? 0u : epoch; const float* ip = PR(P_INITPOSE) + 7 * b;
      float e[3], dq[4], qo[4];
      for (int i = 0; i < 3; i++) ST(S_BPOS)[3 * b + i] = ip[i] + (urand(C.seed, (uint32_t)C.env_id, ep, (uint32_t)(k * 8 + i)) - 0.5f) * fa[i];
      for (int i = 0; i < 3; i++) e[i] = (urand(C.seed, (uint32_t)C.env_id, ep, (uint32_t)(k * 8 + 3 + i)) - 0.5f) * fa[3 + i];
      q_from_euler(dq, e); q_mul(qo, ip + 3, dq); for (int i = 0; i < 4; i++) ST(S_BQUAT)[4 * b + i] = qo[i];
      v_set(ST(S_BVEL) + 3 * b, 0, 0, 0); v_set(ST(S_BOMEGA) + 3 * b, 0, 0, 0);
    } else if (op[0] == OP_VIS_RANDOMIZE) {             // visual_randomizer.py:41-46: a new look for the model on every reset - here a random
      // colour per visual shape of the body (the reference picks a random texture of a dataset it downloads; out of scope)
      for (int v = 0; v < sc.nv; v++) if (gc(sc.vis_i)[DG_VIS_I_W * v + 3] == ia[0])
        for (int i = 0; i < 3; i++) PR(P_COLOR)[3 * v + i] = urand(C.seed, (uint32_t)C.env_id, epoch, (uint32_t)(k * 8 + 128 + 3 * v + i));
    } else if (op[0] == OP_DYN_RANDOMIZE) {             // dynamics_randomizer.py:24-32 (log-uniform on nominal values)
      int b = ia[0]; const int* bi = gc(sc.body_i) + DG_BODY_I_W * b;
      for (int l = -1; l < bi[2]; l++) {
        int f = l < 0 ? b : sc.nb + bi[1] + l; int d = l < 0 ? -1 : shc(C.link_i)[DG_LINK_I_W * (bi[1] + l) + 3];
        if (l >= 0 && d < 0) continue;
        if (l < 0 && bi[4] > 0) continue;
        float u1 = urand(C.seed, (uint32_t)C.env_id, epoch, (uint32_t)(k * 8 + 64 + 2 * (l + 1)));
        float u2 = urand(C.seed, (uint32_t)C.env_id, epoch, (uint32_t)(k * 8 + 65 + 2 * (l + 1)));
        float ms = expf(logf(fa[0]) + u1 * (logf(fa[1]) - logf(fa[0]))), ds = expf(logf(fa[2]) + u2 * (logf(fa[3]) - logf(fa[2])));
        PR(P_MASS)[f] = gc(sc.param_def)[DG_PO(C.sc, P_MASS) + f] * ms;
        for (int i = 0; i < 3; i++) PR(P_INERTIA)[3 * f + i] = gc(sc.param_def)[DG_PO(C.sc, P_INERTIA) + 3 * f + i] * ms;
        // fa[6]: nominal joint damping for joints whose URDF gives none (UR5: 0 - scaling it would do nothing; extension key)
        if (d >= 0) { const float nom = gc(sc.param_def)[DG_PO(C.sc, P_JDAMP) + d]; PR(P_JDAMP)[d] = (nom > 0.f ? nom : fa[6]) * ds; }
      }
      // extension key friction_range (BASELINE.json config 5, SURVEY 8d: lateral friction U[0.5, 1.25] per environment): one draw
      // per body and reset, every collision shape of the body gets it
      if (fa[5] > 0.f) {
        const float u3 = urand(C.seed, (uint32_t)C.env_id, epoch, (uint32_t)(k * 8 + 63));
        const float fr = fa[4] + u3 * (fa[5] - fa[4]);
        for (int s2 = 0; s2 < sc.ns; s2++) if (gc(sc.shape_i)[DG_SHAPE_I_W * s2] == b) PR(P_FRICTION)[s2] = fr;
      }
    }
  }
  ST(S_RESETS)[0] += 1.f;
}

// ------------------------------------------------------------------ the phase schedule -------------------------
// A block advances E environments at once, T lanes each.  Thread t is lane (t / E) of environment (t % E): the 32
// threads of a warp are the SAME lane index of 32 different environments, so a phase in which only a few lanes per
// environment have work (one lane per body, one per IK op ...) runs on a few FULL warps while the other warps wait
// at the barrier without issuing anything.  Phases are separated by block barriers; therefore every decision that
// changes the number of barriers (narrow-phase rounds, "is there any contact", "is any pair of bodies coupled") is
// taken block-uniformly with block_any().  Environments without work in this launch (tail of the batch, reset mask
// off) have C.active == false: they skip the phase bodies but keep the barriers.  T == 1 needs no barriers at all.
// The CPU emulation runs one environment at a time, lane after lane - exactly the barrier semantics.
#if defined(__CUDA_ARCH__)
// (with C.dbg set, thread 0 of every block adds the cycles of each phase, barrier included, to its slot of the debug table)
#define DG_PHASE(call) do { const long long t0_ = C.dbg ? clock64() : 0; if (C.active) { call; } if (nt > 1) __syncthreads(); \
                            if (C.dbg && threadIdx.x == 0) C.dbg[(size_t)blockIdx.x * 64 + (__LINE__ & 63)] += (unsigned long long)(clock64() - t0_); } while (0)
#define DG_LANE_ARGS int ln
DG_HD bool block_any(bool p, int nt) { return nt > 1 ? (__syncthreads_or(p ? 1 : 0) != 0) : p; }
#else
#define DG_PHASE(call) do { for (int ln = 0; ln < nt; ln++) { call; } } while (0)
#define DG_LANE_ARGS int
DG_HD bool block_any(bool p, int) { return p; }
#endif
#define HDRV(k) (C.active ? WSI(C)[SC.W_HDR + (k)] : 0)

// One sub-step up to and including the contact solve of every environment that is not deferred to the sweep kernel
DG_NOINLINE DG_FN void physics_pre(const Env& C, int nt, float h, DG_LANE_ARGS) {
  const DevScene& sc = SC;
  DG_PHASE(phase_dynamics(C, ln, nt, h));
  DG_PHASE(phase_shape_world(C, ln, nt));
  if (sc.npair > 0) {
    DG_PHASE(phase_broad(C, ln, nt));
    DG_PHASE(phase_count_survivors(C, ln, nt));
    for (int rnd = 0; block_any(rnd * nt < HDRV(WH_NSURV), nt); rnd++) {
      DG_PHASE(phase_narrow(C, ln, nt, rnd));
      DG_PHASE(phase_append(C, ln, nt));
    }
  }
  DG_PHASE(phase_minv(C, ln, nt));
  DG_PHASE(phase_unit_rows(C, ln, nt, h));
  if (sc.ncons == 0 && !block_any(HDRV(WH_NCROW) > 0, nt)) {
    DG_PHASE(phase_pgs_unit(C, ln, nt, 0, sc.iters));
  } else {
    DG_PHASE(phase_contact_rows(C, ln, nt, h));
#if defined(__CUDA_ARCH__)
    if (!C.active && ln == 0) { WSI(C)[sc.W_HDR + WH_RS_R] = 0; WSI(C)[sc.W_HDR + WH_RS_NEED] = 0; WSI(C)[sc.W_HDR + WH_RS_DEFER] = 0; }   // slots without an environment never wrote their header
#endif
    DG_PHASE(phase_rs_plan(C, ln, nt));
    DG_PHASE(phase_rs_setup(C, ln, nt));
    // environments with contacts: solved in row space (A is built here; swept below by the team, or - deferred - by a warp of the
    // sweep kernel); contact-free ones keep the register-resident per-body sweeps.  (WH_RS_R == 0 with contacts: dv-space sweeps,
    // solver == 0 / too many rows)
    DG_PHASE(if (HDRV(WH_RS_R) > 0) { if (HDRV(WH_RS_DEFER) == 0) phase_rs_build(C, ln, nt); }   // (deferred: the sweep kernel builds its own columns of A)
             else if (HDRV(WH_COUPLED) == 0) { if (HDRV(WH_NCROW) > 0) phase_pgs_full(C, ln, nt); else phase_pgs_unit(C, ln, nt, 0, sc.iters); });
    if (sc.solver == 1 && nt > 1 && block_any(HDRV(WH_RS_R) > 0 && HDRV(WH_RS_DEFER) == 0, nt)) {
#if defined(__CUDA_ARCH__)
      const long long t0_ = C.dbg ? clock64() : 0;
#if defined(DG_STEP_T)
      rs_solve_block<DG_STEP_T>(C);
#endif
      __syncthreads();
      if (C.dbg && threadIdx.x == 0) C.dbg[(size_t)blockIdx.x * 64 + (__LINE__ & 63)] += (unsigned long long)(clock64() - t0_);
#else
      DG_PHASE(if (ln == 0 && HDRV(WH_RS_R) > 0) rs_solve_serial(C, nt));
#endif
      DG_PHASE(if (HDRV(WH_RS_R) > 0 && HDRV(WH_RS_DEFER) == 0) phase_rs_finish(C, ln, nt));
    }
    if (block_any(HDRV(WH_COUPLED) != 0 && HDRV(WH_RS_R) == 0, nt)) {   // dv-space, coupled bodies: lock-step sweeps
      for (int it = 0; it < sc.iters; it++) {
        DG_PHASE(if (HDRV(WH_COUPLED) != 0 && HDRV(WH_RS_R) == 0) phase_pgs_unit(C, ln, nt, it, it + 1));
        DG_PHASE(if (HDRV(WH_COUPLED) != 0 && HDRV(WH_RS_R) == 0) phase_pgs_contact(C, ln, nt));
      }
    }
  }
}
// ... and the rest of it: impulses of the deferred environments (swept by the sweep kernel in between) folded into dv, integration
DG_NOINLINE DG_FN void physics_post(const Env& C, int nt, float h, DG_LANE_ARGS) {
  // (deferred environments: the sweep kernel has folded the impulses into dv and the unit-row records of the carried workspace)
  DG_PHASE(phase_integrate(C, ln, nt, h));
  if (SC.sem & SEM_WRENCH_FIRST_SUBSTEP) DG_PHASE(phase_next_substep(C, ln, nt));
}
// p.stepSimulation() (diy_gym.py:146,207); nsub = 0 only refreshes the link cache
DG_NOINLINE DG_FN void run_physics(const Env& C, int nt, int nsub, int clear_forces, DG_LANE_ARGS) {
  const DevScene& sc = SC;
  float h = sc.dt / (float)sc.substeps;
  DG_PHASE(phase_load(C, ln, nt));
  for (int sub = 0; sub < nsub; sub++) {
#if defined(__CUDA_ARCH__)
    physics_pre(C, nt, h, ln); physics_post(C, nt, h, ln);
#else
    physics_pre(C, nt, h, 0); physics_post(C, nt, h, 0);
#endif
  }
  DG_PHASE(phase_final_kin(C, ln, nt));
  DG_PHASE(phase_store(C, ln, nt, clear_forces));
}
#if defined(__CUDA_ARCH__)
// One DIYGym.step cut into kernel launches around the sweep kernel (dg_kernels.cu, "split schedule"):
//   ST_ACT  add-on update + state row -> workspace      ST_PRE  physics_pre of one sub-step
//   ST_POST physics_post of one sub-step                ST_END  link cache + state row back, sensors / rewards / terminals
//   ST_LOAD: state row -> workspace without add-on update: the hot-start steps of DIYGym.reset (the reset hooks themselves run as
//   one fused launch with Env::no_hot set).  (Calling phase_reset_ops + run_physics from here as well made nvcc 12.9 emit a step
//   kernel whose IK returned its input - 10 MB more code per object, results wrong on the B200, right in the g++ build.)
// The hot workspace travels between launches through the per-environment carry buffer (ST_SAVEC / ST_LOADC, done by the
// kernel around this call); the cold workspace is per environment anyway.
DG_FN void run_env_step_stages(const Env& C, int nt, int stages, int ln) {
  const DevScene& sc = SC;
  const float h = sc.dt / (float)sc.substeps;
  if (stages & ST_ACT) { DG_PHASE(phase_actions(C, ln, nt)); DG_PHASE(phase_load(C, ln, nt)); }
  if (stages & ST_LOAD) { DG_PHASE(phase_load(C, ln, nt)); }                                        // a hot-start step has no add-on update
  if (stages & ST_POST) physics_post(C, nt, h, ln);
  if (stages & ST_PRE) physics_pre(C, nt, h, ln);
  if (stages & ST_END) { DG_PHASE(phase_final_kin(C, ln, nt)); DG_PHASE(phase_store(C, ln, nt, 1)); DG_PHASE(phase_observe(C, ln, nt)); }
}
#endif

// DIYGym.step for one environment
DG_FN void run_env_step(const Env& C, int nt, DG_LANE_ARGS) {
#if defined(__CUDA_ARCH__)
  DG_PHASE(phase_actions(C, ln, nt));
  run_physics(C, nt, SC.substeps, 1, ln);
  DG_PHASE(phase_observe(C, ln, nt));
#else
  DG_PHASE(phase_actions(C, ln, nt));
  run_physics(C, nt, SC.substeps, 1, 0);
  DG_PHASE(phase_observe(C, ln, nt));
#endif
}
// DIYGym.observe / reward / is_terminal from the state rows as they are (diy_gym.py:211-222): refreshes the link cache the
// sensors read (no physics), then evaluates every sensor / reward / terminal op
DG_FN void run_env_observe(const Env& C, int nt, DG_LANE_ARGS) {
#if defined(__CUDA_ARCH__)
  run_physics(C, nt, 0, 0, ln);
#else
  run_physics(C, nt, 0, 0, 0);
#endif
  DG_PHASE(phase_observe(C, ln, nt));
}
// DIYGym.reset for one environment
DG_FN void run_env_reset(const Env& C, int nt, DG_LANE_ARGS) {
#if defined(__CUDA_ARCH__)
  DG_PHASE(phase_reset_ops(C, ln, nt));
  run_physics(C, nt, 0, 0, ln);
  for (int i = 0; i < (C.no_hot ? 0 : SC.hot_start); i++) run_physics(C, nt, SC.substeps, 1, ln);
  DG_PHASE(phase_observe(C, ln, nt));
#else
  DG_PHASE(phase_reset_ops(C, ln, nt));
  run_physics(C, nt, 0, 0, 0);
  for (int i = 0; i < SC.hot_start; i++) run_physics(C, nt, SC.substeps, 1, 0);
  DG_PHASE(phase_observe(C, ln, nt));
#endif
}

// The Env of a kernel that only reads state rows (camera, ray_sensor, IK query): the scene, the row st and the scene's link tables;
// every other member null / zero.  (At the end of the file: the phase-timing keys of DG_PHASE are source lines.)
DG_HD Env row_env(const DevScene& sc, float* st) {
  Env C{};
  C.sc = &sc; C.st = st; C.link_i = sc.link_i; C.link_f = sc.link_f; C.link_x = sc.link_x;
  return C;
}

}  // namespace dg
