"""fp64 numpy restatement of the inverse-kinematics query (csrc/dg_ik.cuh over ik_solve* of csrc/dg_env.cuh): damped least
squares on the URDF frame of one link, in the coordinates of the base, with the seed, null-space lists, iterations and threshold
as arguments.  Forward kinematics is the plain URDF transform product of tests/helpers.py urdf_kinematics, moved from the
body's spawn pose to the state row's base pose; nothing is read from the compiled link tables.

Per iteration, at the current q: position error e_p = t_p - p(q) and, with an orientation, e_o = axis * angle of
t_q conj(q(q)) (angle wrapped into [-pi, pi]); the loop stops before an iteration whose q already had |e_p| <= threshold.
  without null-space lists: dq = (J^T J + ik_damping I)^-1 J^T e
  with them:                dq = J^T (J J^T + ik_null_lambda_sq I)^-1 (e - J n) + n,
                            n_i = 0.001 (rest_i - q0_i) + 10 (upper_i - q0_i) / range_i if q0_i > upper_i (lower alike), from the seed q0
dq is scaled so that its largest entry is at most 45 degrees.  err: |e_p| and the remaining rotation angle at the returned q."""
import numpy as np

from diy_gym_b200.compiler.mathutil import Transform, quat_conj, quat_mul, quat_to_mat
from tests.helpers import urdf_kinematics


def _frames(sc, body, q, base_pos, base_quat):
    """URDF link frames, joint axes and joint origins of `body` at q, for the base COM at (base_pos, base_quat)."""
    b = sc.bodies[body]
    Tl, _, axes, orgs = urdf_kinematics(sc, q, body)
    move = Transform(base_pos, base_quat) * Transform(b.base_pos, b.base_quat).inverse()
    R = quat_to_mat(move.q)
    return ([move * T for T in Tl], [None if a is None else R @ a for a in axes], [None if o is None else move.apply(o) for o in orgs])


def _rotation_error(tq, qc):
    dq = quat_mul(tq, quat_conj(qc))
    vn = np.linalg.norm(dq[:3])
    ang = 2 * np.arctan2(vn, dq[3])
    ax = np.array([1., 0., 0.]) if vn * vn < 10 * 2.220446049250313e-16 else dq[:3] / vn
    if ang > np.pi:
        ang -= 2 * np.pi
    elif ang < -np.pi:
        ang += 2 * np.pi
    return ax * ang


def ik(sc, state, body, link, tpos, torn=None, q0=None, limits=None, iters=None, threshold=None):
    """(q [n_dof], err [2]) for link `link` (joint index) of `body`, from one state row; limits: (lower, upper, range, rest)."""
    b, h = sc.bodies[body], sc.hdr
    nd, d0 = b.n_dofs, b.dof_start
    state = np.asarray(state, np.float64)
    iters = h['ik_iters'] if iters is None else iters
    threshold = sc.hdr_f['ik_threshold'] if threshold is None else threshold
    q = (state[h['S_Q'] + d0:h['S_Q'] + d0 + nd] if q0 is None else np.asarray(q0, np.float64)).copy()
    bp = state[h['S_BPOS'] + 3 * body:h['S_BPOS'] + 3 * body + 3]
    bq = state[h['S_BQUAT'] + 4 * body:h['S_BQUAT'] + 4 * body + 4]
    bq = bq / np.linalg.norm(bq)
    tpos = np.asarray(tpos, np.float64)
    tq = None if torn is None else np.asarray(torn, np.float64) / np.linalg.norm(torn)
    nullv = np.zeros(nd)
    if limits is not None:
        lo, up, rg, rest = [np.asarray(v, np.float64) for v in limits]
        nullv = 0.001 * (rest - q) + np.where(q > up, 10 * (up - q) / rg, 0) + np.where(q < lo, 10 * (lo - q) / rg, 0)
    L = b.links
    chain, k = [], link + 1
    while k > 0:
        chain.append(k)
        k = L[k]['parent']
    dof_of, d = {}, 0
    for k in range(1, len(L)):
        if L[k]['joint']['type'] != 'fixed':
            dof_of[k] = d
            d += 1
    m = 3 if tq is None else 6

    def residual(q):
        T, axes, orgs = _frames(sc, body, q, bp, bq)
        e = np.zeros(m)
        e[:3] = tpos - T[link + 1].p
        if tq is not None:
            e[3:] = _rotation_error(tq, T[link + 1].q)
        return e, T, axes, orgs

    diff = np.inf
    for _ in range(iters):
        if not diff > threshold:
            break
        e, T, axes, orgs = residual(q)
        diff = np.linalg.norm(e[:3])
        J = np.zeros((m, nd))
        for k in chain:
            if k not in dof_of:
                continue
            c = dof_of[k]
            if L[k]['joint']['type'] == 'prismatic':
                J[:3, c] = axes[k]
            else:
                J[:3, c] = np.cross(axes[k], T[link + 1].p - orgs[k])
                if m == 6:
                    J[3:, c] = axes[k]
        if limits is None:
            dq = np.linalg.solve(J.T @ J + sc.hdr_f['ik_damping'] * np.eye(nd), J.T @ e)
        else:
            dq = J.T @ np.linalg.solve(J @ J.T + sc.hdr_f['ik_null_lambda_sq'] * np.eye(m), e - J @ nullv) + nullv
        mx = np.abs(dq).max()
        if mx > np.pi / 4:
            dq *= np.pi / 4 / mx
        q = q + dq
    e, T, _, _ = residual(q)
    ang = 0.0
    if tq is not None:
        dq = quat_mul(tq, quat_conj(T[link + 1].q))
        ang = 2 * np.arctan2(np.linalg.norm(dq[:3]), abs(dq[3]))
    return q, np.array([np.linalg.norm(e[:3]), ang])


def fk(sc, state, body, link, q):
    """World pose (position, xyzw) of the URDF frame of link `link` of `body` at q, with the state row's base pose."""
    h = sc.hdr
    state = np.asarray(state, np.float64)
    bp = state[h['S_BPOS'] + 3 * body:h['S_BPOS'] + 3 * body + 3]
    bq = state[h['S_BQUAT'] + 4 * body:h['S_BQUAT'] + 4 * body + 4]
    T = _frames(sc, body, np.asarray(q, np.float64), bp, bq / np.linalg.norm(bq))[0][link + 1]
    return T.p, T.q
