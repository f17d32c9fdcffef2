"""fp64 numpy reference of the dynamics queries (Model.jacobian / mass_matrix / inverse_dynamics, csrc/dg_dyn.cuh), written
from the compiled scene tables plus one state row and one parameter row.

It shares the conventions of the kernel (generalized velocity nu = [omega_base, v_base, qd] for a floating base, qd for a fixed
one; world axes) but not its algorithm: the kernel gets tau from one recursive Newton-Euler pass, this reference forms it as
    tau = M qdd + sum_k Jv_k^T m_k (Jdot_v,k nu - g) + Jw_k^T (I_k Jdot_w,k nu + omega_k x I_k omega_k)
with the Jacobian time derivatives taken by central differences of the Jacobians along the motion (joints q +- h qd, base moved by
+- h v and rotated by exp(+- h [omega]x)).  TEST INFRASTRUCTURE: the product never uses it."""
import numpy as np

from diy_gym_b200.compiler.mathutil import quat_to_mat


def _rot(axis, ang):
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def n_coords(sc, body):
    b = sc.bodies[body]
    return b.n_dofs + (6 if b.kind == 2 else 0)


def kinematics(sc, body, q, Rb, cb):
    """Per link record (0 = base, k + 1 = link k): world rotation and COM, and the columns (w, u, o) of every generalized
    coordinate with the set of columns that move each link."""
    b = sc.bodies[body]
    LI, LF = sc.sec['LINK_I'], sc.sec['LINK_F']
    fb = 6 if b.kind == 2 else 0
    n = fb + b.n_dofs
    R, C, cols = [Rb], [cb], [None] * n
    moved = [set(range(6)) if fb else set()]
    for i in range(fb):
        cols[i] = (np.eye(3)[i], np.zeros(3), cb) if i < 3 else (np.zeros(3), np.eye(3)[i - 3], np.zeros(3))
    for k in range(b.n_links):
        gl = b.link_start + k
        li, lf = LI[gl], np.asarray(LF[gl], float)
        p = 0 if li[1] < 0 else li[1] - b.link_start + 1
        R0, e, d, a = quat_to_mat(lf[0:4]), lf[4:7], lf[7:10], lf[10:13]
        c = fb + b.joint_dof[k] if b.joint_dof[k] >= 0 else -1
        qk = q[b.joint_dof[k]] if c >= 0 else 0.0
        if li[2] == 1:
            Rrel = R0 @ _rot(a, qk)
            r = e + Rrel @ d
        elif li[2] == 2:
            Rrel, r = R0, e + R0 @ (d + a * qk)
        else:
            Rrel, r = R0, e + R0 @ d
        R.append(R[p] @ Rrel)
        C.append(C[p] + R[p] @ r)
        s, o = R[-1] @ a, C[-1] - R[-1] @ d
        moved.append(moved[p] | ({c} if c >= 0 else set()))
        if c >= 0:
            cols[c] = (s, np.zeros(3), o) if li[2] == 1 else (np.zeros(3), s, np.zeros(3))
    return R, C, cols, moved


def link_jacobian(cols, moved_k, P):
    n = len(cols)
    Jv, Jw = np.zeros((3, n)), np.zeros((3, n))
    for c in moved_k:
        w, u, o = cols[c]
        Jv[:, c], Jw[:, c] = np.cross(w, P - o) + u, w
    return Jv, Jw


def _row(sc, state, param, body):
    h, b = sc.hdr, sc.bodies[body]
    st, pr = np.asarray(state, float), np.asarray(param, float)
    q = st[h['S_Q'] + b.dof_start:h['S_Q'] + b.dof_start + b.n_dofs]
    qd = st[h['S_QD'] + b.dof_start:h['S_QD'] + b.dof_start + b.n_dofs]
    if b.kind == 2:
        qd = np.r_[st[h['S_BOMEGA'] + 3 * body:h['S_BOMEGA'] + 3 * body + 3], st[h['S_BVEL'] + 3 * body:h['S_BVEL'] + 3 * body + 3], qd]
    Rb = quat_to_mat(st[h['S_BQUAT'] + 4 * body:h['S_BQUAT'] + 4 * body + 4])
    cb = st[h['S_BPOS'] + 3 * body:h['S_BPOS'] + 3 * body + 3].copy()
    frames = [body] + [sc['nb'] + b.link_start + k for k in range(b.n_links)]
    m = pr[h['P_MASS'] + np.array(frames)]
    I = np.stack([pr[h['P_INERTIA'] + 3 * f:h['P_INERTIA'] + 3 * f + 3] for f in frames])
    if b.kind != 2:
        m = m.copy()
        m[0] = 0.0
    return q, qd, Rb, cb, m, I


def dynamics(sc, state, param, body, link=-1, point=(0., 0., 0.), q=None, qd=None, qdd=None, h=1e-5):
    """(J [6, n] linear rows first, M [n, n], tau [n]) of body `body` for one state row and one parameter row (fp64)."""
    b = sc.bodies[body]
    q0, qd0, Rb, cb, m, I = _row(sc, state, param, body)
    q = q0 if q is None else np.asarray(q, float)
    nu = qd0 if qd is None else np.asarray(qd, float)
    n = n_coords(sc, body)
    qdd = np.zeros(n) if qdd is None else np.asarray(qdd, float)
    fb = 6 if b.kind == 2 else 0
    g = np.array([sc.hdr_f['gx'], sc.hdr_f['gy'], sc.hdr_f['gz']])

    def jacs(t):
        qt = q + t * nu[fb:]
        if fb:
            w = nu[0:3]
            wn = np.linalg.norm(w)
            Rt = (_rot(w / wn, t * wn) if wn > 0 else np.eye(3)) @ Rb
            ct = cb + t * nu[3:6]
        else:
            Rt, ct = Rb, cb
        R, C, cols, moved = kinematics(sc, body, qt, Rt, ct)
        return R, C, [link_jacobian(cols, moved[k], C[k]) for k in range(len(C))], cols, moved

    R, C, J0, cols, moved = jacs(0.0)
    _, _, Jp, _, _ = jacs(h)
    _, _, Jm, _, _ = jacs(-h)
    M, tau = np.zeros((n, n)), np.zeros(n)
    for k in range(len(C)):
        Jv, Jw = J0[k]
        Iw = R[k] @ np.diag(I[k]) @ R[k].T
        M += m[k] * Jv.T @ Jv + Jw.T @ Iw @ Jw
        om = Jw @ nu
        av = (Jp[k][0] - Jm[k][0]) @ nu / (2 * h)
        aw = (Jp[k][1] - Jm[k][1]) @ nu / (2 * h)
        tau += Jv.T @ (m[k] * (av - g)) + Jw.T @ (Iw @ aw + np.cross(om, Iw @ om))
    tau += M @ qdd
    P = C[link + 1] + R[link + 1] @ np.asarray(point, float)
    Jv, Jw = link_jacobian(cols, moved[link + 1], P)
    return np.vstack([Jv, Jw]), M, tau

