"""Shared test helpers: scene construction and an *independent* numpy rigid-body reference
(world-frame Jacobian mass matrix + potential-energy gradient) used to pin the oracle's ABA."""
import numpy as np

from diy_gym_b200.assets import resolve_model
from diy_gym_b200.compiler.mathutil import Transform, quat_rotate, quat_to_mat
from diy_gym_b200.compiler.scene import SceneBuilder


def build_single(model, world=None, **kw):
    sb = SceneBuilder(**(world or {}))
    sb.add_body('m', resolve_model(model), **kw)
    return sb.finalize()


def free_dynamics(w, sc):
    """Switch off motors and every damping term of an OracleWorld."""
    w.s('S_MMAXF', sc['nd'])[:] = 0
    w.p('P_LINDAMP', sc['nb'])[:] = 0
    w.p('P_ANGDAMP', sc['nb'])[:] = 0
    w.p('P_JDAMP', sc['nd'])[:] = 0


def urdf_kinematics(sc, q, body=0):
    """World transforms of every URDF link frame / COM frame as a plain product of the URDF <origin>s."""
    b = sc.bodies[body]
    L, s = b.links, b.scale
    Tl = [None] * len(L)
    Tl[0] = Transform(b.base_pos, b.base_quat) * Transform.from_xyz_rpy(np.array(L[0]['inertial_xyz']) * s,
                                                                       L[0]['inertial_rpy']).inverse()
    axes, orgs, coms, dof = [None] * len(L), [None] * len(L), [None] * len(L), 0
    for k in range(1, len(L)):
        j = L[k]['joint']
        T = Tl[L[k]['parent']] * Transform.from_xyz_rpy(np.array(j['xyz']) * s, j['rpy'])
        if j['type'] in ('revolute', 'continuous'):
            ax = np.array(j['axis']) / np.linalg.norm(j['axis'])
            axes[k], orgs[k] = quat_rotate(T.q, ax), T.p.copy()
            T = T * Transform((0, 0, 0), np.r_[ax * np.sin(q[dof] / 2), np.cos(q[dof] / 2)])
            dof += 1
        elif j['type'] == 'prismatic':
            ax = np.array(j['axis']) / np.linalg.norm(j['axis'])
            axes[k] = quat_rotate(T.q, ax)
            T = T * Transform(ax * q[dof])
            dof += 1
        Tl[k] = T
    for k in range(len(L)):
        coms[k] = Tl[k] * Transform.from_xyz_rpy(np.array(L[k]['inertial_xyz']) * s, L[k]['inertial_rpy'])
    return Tl, coms, axes, orgs


def mass_matrix_gravity_energy(sc, w, q, qd=None, g=(0, 0, -9.81), body=0):
    """M(q), generalized gravity G(q) (M qdd + G = tau at qd = 0) and total energy, fixed-base bodies."""
    b = sc.bodies[body]
    L, nd = b.links, b.n_dofs
    Tl, coms, axes, orgs = urdf_kinematics(sc, q, body)
    mass = w.p('P_MASS', sc['nframes'])
    inert = w.p('P_INERTIA', 3 * sc['nframes']).reshape(-1, 3)
    d, dof_of = 0, [-1] * len(L)
    for k in range(1, len(L)):
        if L[k]['joint']['type'] != 'fixed':
            dof_of[k] = d
            d += 1
    M, G, pot = np.zeros((nd, nd)), np.zeros(nd), 0.0
    for k in range(1, len(L)):
        f = b.frame(k - 1)
        m, Iw = mass[f], None
        R = quat_to_mat(coms[k].q)
        Iw = R @ np.diag(inert[f]) @ R.T
        Jv, Jw = np.zeros((3, nd)), np.zeros((3, nd))
        a = k
        while a > 0:
            if dof_of[a] >= 0:
                if L[a]['joint']['type'] == 'prismatic':
                    Jv[:, dof_of[a]] = axes[a]
                else:
                    Jw[:, dof_of[a]] = axes[a]
                    Jv[:, dof_of[a]] = np.cross(axes[a], coms[k].p - orgs[a])
            a = L[a]['parent']
        M += m * Jv.T @ Jv + Jw.T @ Iw @ Jw
        G += -Jv.T @ (m * np.array(g))
        pot += -m * np.dot(g, coms[k].p)
    energy = pot + (0.5 * qd @ M @ qd if qd is not None else 0.0)
    return M, G, energy


# ---------------------------------------------------------------- strict single-step parity protocol -----------------
def strict_single_step_parity(env, n_envs, steps, seed=4321, presteps=3, action_scale=None):
    """BASELINE.json north_star bar, exactly: every step BOTH arms start from the same fp32-rounded state row, take the same
    action, and the states after ONE DIYGym.step are compared environment by environment:
        |dq|  <= 1e-4 * max|q|            |dqd| <= 1e-4 * max(max|qd|, 1e-2)
        base position / quaternion / linear / angular velocity of every body: 1e-4 relative to the largest entry of the
        section (floors: 1e-2 for the twists, as for qd)
    `env` is a DIYGym on either world (CUDA through the C ABI, or the CPU build of the kernel source in tests/emul).
    Returns the per-step records (worst errors, bars, contact counts of the oracle) - the caller asserts."""
    import torch
    from oracle.oracle import OracleWorld
    w, sc, h = env.world, env.scene, env.scene.hdr
    nd, nb = sc['nd'], sc['nb']
    cuda = w.state.is_cuda
    if action_scale is None:
        from bench import action_ranges
        lo, hi = action_ranges(env)
    else:
        lo, hi = -action_scale * np.ones(max(sc['n_act'], 1))[:sc['n_act']], action_scale * np.ones(max(sc['n_act'], 1))[:sc['n_act']]
    oracles = [OracleWorld(sc, seed=seed, env_id=i) for i in range(n_envs)]
    rng = np.random.default_rng(seed)
    for i, o in enumerate(oracles):
        o.env_reset()
        for _ in range(presteps + i % 4):      # decorrelate the environments
            o.env_step(rng.uniform(lo, hi))
    recs = []
    ncon_prev = np.array([len(o.contacts()) for o in oracles])
    for k in range(steps):
        st = np.stack([o.state for o in oracles]).astype(np.float32)
        w.state.copy_(torch.from_numpy(st))
        w.param.copy_(torch.from_numpy(np.stack([o.param for o in oracles]).astype(np.float32)))
        for i, o in enumerate(oracles):
            o.state[:] = st[i]
        a = rng.uniform(lo, hi, (n_envs, max(w.n_act, 1))).astype(np.float32)[:, :w.n_act]
        if w.n_act:
            w.action.copy_(torch.from_numpy(a))
        w.step()
        if cuda:
            torch.cuda.synchronize()
        outs = [o.env_step(a[i].astype(np.float64)) for i, o in enumerate(oracles)]
        ncon = np.array([len(o.contacts()) for o in oracles])
        sg = w.state.cpu().numpy().astype(np.float64)
        so = np.stack([o.state for o in oracles])
        rec = {'step': k, 'contacts': ncon, 'err': {}, 'bar': {}, 'err_free': {}}
        free = (ncon == 0) & (ncon_prev == 0)   # contact-free: no contact in the oracle before or after the step
        ncon_prev = ncon
        for key, nm, n, floor in (('q', 'S_Q', nd, 0.0), ('qd', 'S_QD', nd, 1e-2), ('base_pos', 'S_BPOS', 3 * nb, 0.0), ('base_quat', 'S_BQUAT', 4 * nb, 0.0),
                                  ('base_vel', 'S_BVEL', 3 * nb, 1e-2), ('base_omega', 'S_BOMEGA', 3 * nb, 1e-2)):
            if n == 0:
                continue
            g, o_ = sg[:, h[nm]:h[nm] + n], so[:, h[nm]:h[nm] + n]
            rec['err'][key] = float(np.abs(g - o_).max())
            rec.setdefault('err_env', {})[key] = np.abs(g - o_).max(axis=1)   # per environment
            rec['err_free'][key] = float(np.abs(g - o_)[free].max()) if free.any() else 0.0
            rec['bar'][key] = 1e-4 * max(float(np.abs(o_).max()), floor)
        rec['obs'] = (w.obs.cpu().numpy().astype(np.float64), np.stack([x[0] for x in outs]))
        rec['rew'] = (w.reward.cpu().numpy().astype(np.float64), np.stack([x[1] for x in outs]))
        rec['term'] = (w.term.cpu().numpy(), np.stack([x[2] for x in outs]))
        recs.append(rec)
    return recs


def golden_mesh(rel):
    """(vertices, lo, hi) of source mesh `rel` from tests/golden/mesh_vertices.npz (tools/make_mesh_golden.py): vertices of the
    mesh that include its extreme ones along each axis, and its bounding box, in the mesh frame."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'mesh_vertices.npz'))
    k = os.path.splitext(os.path.basename(rel))[0]
    return g['verts_' + k], g['lo_' + k], g['hi_' + k]


def write_mesh(path, verts):
    """Writes a vertex cloud as a binary STL (triangles of consecutive vertices, the last one repeated to fill the last
    triangle) or as a COLLADA file with one position source, chosen by the extension."""
    import struct
    v = np.asarray(verts, np.float64)
    if path.endswith('.dae'):
        floats = ' '.join('%.17g' % x for x in v.reshape(-1))
        with open(path, 'w') as f:
            f.write('<?xml version="1.0"?>\n<COLLADA xmlns="http://www.collada.org/2005/11/COLLADASchema" version="1.4.1">'
                    '<library_geometries><geometry id="g"><mesh><source id="g-positions"><float_array id="g-positions-array" '
                    'count="%d">%s</float_array></source><vertices id="g-vertices"><input semantic="POSITION" source="#g-positions"/>'
                    '</vertices></mesh></geometry></library_geometries></COLLADA>\n' % (v.size, floats))
        return
    v = np.concatenate([v, np.repeat(v[-1:], -len(v) % 3, axis=0)]).astype('<f4').reshape(-1, 9)
    with open(path, 'wb') as f:
        f.write(b'\0' * 80 + struct.pack('<I', len(v)))
        for tri in v:
            f.write(struct.pack('<3f', 0, 0, 0) + tri.tobytes() + struct.pack('<H', 0))
