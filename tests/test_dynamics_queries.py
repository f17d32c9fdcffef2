"""Batched rigid-body dynamics queries of a Model: jacobian / mass_matrix / inverse_dynamics (pybullet's calculateJacobian /
calculateMassMatrix / calculateInverseDynamics, csrc/dg_dyn.cuh + dg_dyn_kernel), apply_joint_torque and disable_motors.

CPU: the fp64 reference (tests/dynamics_reference.py) is pinned by known answers and by the oracle's forward dynamics; the g++
build of dg_dyn.cuh (tests/emul/dyn_emul.py) is checked against it on the example scenes; the host layer runs on the emulated
world, including the reference's admittance controller written as a user add-on on these queries.  GPU: the same checks on the
kernel, plus J nu against the step kernel's link-velocity cache, side effects and streams."""
import os

import numpy as np
import pytest
import torch

from diy_gym_b200 import spaces
from diy_gym_b200.addons.addon import Addon, AddonFactory
from diy_gym_b200.compiler.mathutil import quat_from_euler, quat_to_mat
from oracle.oracle import OracleWorld
from tests.dynamics_reference import dynamics, n_coords
from tests.helpers import build_single, free_dynamics, mass_matrix_gravity_energy, urdf_kinematics

EX = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'examples')
ARMS = ['ur5/ur5_robot.urdf', 'jaco/j2s7s300_standalone.urdf']
SCENES = [('ur_high_5', 'ur_high_5_randomised'), ('from_the_readme', 'from_the_readme'), ('r2d2_maze', 'r2d2_maze'),
          ('drone_pilot', 'drone_pilot')]


def _valid_q(model, rng, nd):
    q = rng.uniform(-1, 1, nd)
    if 'jaco' in model:   # away from the limits of the Jaco's joints 2, 4, 6 and of its fingers
        q[[1, 3, 5]] += 3.0
        q[7:] = rng.uniform(0.2, 1.8, 3)
    if 'r2d2' in model:   # inside the gripper's limits: extension [-0.38, 0], fingers [0, 0.548]
        q[4], q[5:7] = rng.uniform(-0.3, -0.1), rng.uniform(0.1, 0.4, 2)
    return q


def _env(folder, name, n, factory=None, path=None):
    from bench import register_example_addons
    from diy_gym_b200 import DIYGym
    register_example_addons()
    return DIYGym(path or os.path.join(EX, folder, name + '.yaml'), num_envs=n, device=0, seed=4321, world_factory=factory)


def _emul_env(folder, name, n=4, path=None):
    from tests.emul.dyn_emul import factory
    return _env(folder, name, n, factory(4), path)


def _models(receptor):
    for m in receptor.models.values():
        yield m
        yield from _models(m)


def _movable(env):
    return [m for m in _models(env) if n_coords(env.scene, m.uid) > 0]


# ---------------------------------------------------------------- (1) the reference, pinned by known answers --------------
@pytest.mark.parametrize('model', ARMS)
def test_reference_fixed_base_mass_matrix_and_gravity_equal_helpers(model):
    sc = build_single(model, fixed_base=True, xyz=(0.1, -0.2, 0.3), quat=quat_from_euler([0.3, -0.2, 0.5]))
    w = OracleWorld(sc)
    nd = sc['nd']
    q = _valid_q(model, np.random.default_rng(0), nd)
    w.s('S_Q', nd)[:] = q
    M0, G0, _ = mass_matrix_gravity_energy(sc, w, q)
    _, M, G = dynamics(sc, w.state, w.param, 0, qd=np.zeros(nd))
    assert np.abs(M - M0).max() <= 1e-10 * np.abs(M0).max()
    assert np.abs(G - G0).max() <= 1e-10 * np.abs(G0).max()


@pytest.mark.parametrize('model', ARMS)
def test_reference_jacobian_equals_shim_and_finite_differences(model):
    from oracle.shim import pybullet as pb
    from diy_gym_b200.assets import resolve_model
    sc = build_single(model, fixed_base=True)
    w = OracleWorld(sc)
    b, nd = sc.bodies[0], sc['nd']
    q = _valid_q(model, np.random.default_rng(1), nd)
    w.s('S_Q', nd)[:] = q
    pb.resetSimulation()
    pb._sim.specs.append(dict(desc=resolve_model(model), scale=1.0, fixed=True, pos=np.zeros(3), quat=np.array([0., 0., 0., 1.]), mass=None))
    pb._sim.ensure()
    point = np.array([0.02, -0.01, 0.05])
    link = b.n_links - 1
    while b.joint_dof[link] < 0 and link > 0:   # the last link a joint moves
        link -= 1
    J = dynamics(sc, w.state, w.param, 0, link, point)[0]
    Jl, Ja = pb.calculateJacobian(0, link, point, list(q), [0.] * nd, [0.] * nd)
    assert np.allclose(J[:3], np.array(Jl), atol=1e-12) and np.allclose(J[3:], np.array(Ja), atol=1e-12)
    # central differences of the URDF transform product: point velocity and rotation rate per unit joint rate
    h = 1e-6
    for c in range(nd):
        dq = np.zeros(nd)
        dq[c] = h
        (_, cp, _, _), (_, cm, _, _) = urdf_kinematics(sc, q + dq), urdf_kinematics(sc, q - dq)
        Pp = cp[link + 1].p + quat_to_mat(cp[link + 1].q) @ point
        Pm = cm[link + 1].p + quat_to_mat(cm[link + 1].q) @ point
        dR = (quat_to_mat(cp[link + 1].q) - quat_to_mat(cm[link + 1].q)) / (2 * h) @ quat_to_mat(urdf_kinematics(sc, q)[1][link + 1].q).T
        om = np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]]) / 2
        assert np.allclose(J[:3, c], (Pp - Pm) / (2 * h), atol=1e-8)
        assert np.allclose(J[3:, c], om, atol=1e-8)


def test_reference_free_rigid_body():
    """A floating body without joints: M = blockdiag(I_world, m 1), tau(qdd = 0) = [omega x I omega, -m g]."""
    sc = build_single('sphere2.urdf', xyz=(0, 0, 1))
    w = OracleWorld(sc)
    rng = np.random.default_rng(2)
    quat = rng.normal(size=4)
    w.s('S_BQUAT', 4)[:] = quat / np.linalg.norm(quat)
    w.p('P_INERTIA', 3)[:] = [0.3, 0.5, 0.7]
    w.s('S_BOMEGA', 3)[:] = rng.uniform(-2, 2, 3)
    w.s('S_BVEL', 3)[:] = rng.uniform(-2, 2, 3)
    m, om = w.p('P_MASS', 1)[0], w.s('S_BOMEGA', 3).copy()
    R = quat_to_mat(w.s('S_BQUAT', 4))
    Iw = R @ np.diag([0.3, 0.5, 0.7]) @ R.T
    J, M, tau = dynamics(sc, w.state, w.param, 0)
    Mref = np.zeros((6, 6))
    Mref[:3, :3], Mref[3:, 3:] = Iw, m * np.eye(3)
    g = np.array([sc.hdr_f['gx'], sc.hdr_f['gy'], sc.hdr_f['gz']])
    assert np.allclose(M, Mref, atol=1e-12)
    assert np.allclose(tau, np.r_[np.cross(om, Iw @ om), -m * g], atol=1e-8)
    assert np.allclose(J, np.eye(6)[[3, 4, 5, 0, 1, 2]], atol=1e-12)


@pytest.mark.parametrize('model', ARMS + ['r2d2.urdf'])
def test_reference_kinetic_energy(model):
    """1/2 nu^T M nu = sum_k 1/2 m_k |v_k|^2 + 1/2 omega_k^T I_k omega_k, with the link twists from finite differences of poses."""
    from tests.dynamics_reference import kinematics, _row
    sc = build_single(model, fixed_base=model != 'r2d2.urdf', xyz=(0, 0, 1))
    w = OracleWorld(sc)
    b, nd = sc.bodies[0], sc['nd']
    n = n_coords(sc, 0)
    rng = np.random.default_rng(3)
    w.s('S_Q', nd)[:] = _valid_q(model, rng, nd)
    nu = rng.uniform(-1, 1, n)
    M = dynamics(sc, w.state, w.param, 0, qd=nu)[1]
    q, _, Rb, cb, m, I = _row(sc, w.state, w.param, 0)
    h, fb = 1e-6, n - nd
    poses = []
    for t in (h, -h):
        Rt, ct = Rb, cb
        if fb:
            from tests.dynamics_reference import _rot
            wn = np.linalg.norm(nu[:3])
            Rt, ct = _rot(nu[:3] / wn, t * wn) @ Rb, cb + t * nu[3:6]
        poses.append(kinematics(sc, 0, q + t * nu[fb:], Rt, ct)[:2])
    R0 = kinematics(sc, 0, q, Rb, cb)[0]
    ke = 0.0
    for k in range(len(R0)):
        v = (poses[0][1][k] - poses[1][1][k]) / (2 * h)
        dR = (poses[0][0][k] - poses[1][0][k]) / (2 * h) @ R0[k].T
        om = np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]]) / 2
        ke += 0.5 * m[k] * v @ v + 0.5 * om @ (R0[k] @ np.diag(I[k]) @ R0[k].T) @ om
    assert abs(0.5 * nu @ M @ nu - ke) <= 1e-8 * ke


# ---------------------------------------------------------------- (2) inverse dynamics inverts the oracle's forward dynamics
@pytest.mark.parametrize('model', ARMS + ['r2d2.urdf'])
def test_inverse_dynamics_inverts_oracle_forward_dynamics(model):
    dt = 1e-7
    floating = model == 'r2d2.urdf'
    sc = build_single(model, world=dict(timestep=dt, substeps=1), fixed_base=not floating, xyz=(0, 0, 2))
    w = OracleWorld(sc)
    nd, n = sc['nd'], n_coords(sc, 0)
    rng = np.random.default_rng(4)
    w.s('S_Q', nd)[:] = _valid_q(model, rng, nd)
    w.s('S_QD', nd)[:] = rng.uniform(-1, 1, nd)
    if floating:
        quat = rng.normal(size=4)
        w.s('S_BQUAT', 4)[:] = quat / np.linalg.norm(quat)
        w.s('S_BOMEGA', 3)[:] = rng.uniform(-1, 1, 3)
        w.s('S_BVEL', 3)[:] = rng.uniform(-1, 1, 3)
    free_dynamics(w, sc)
    w.refresh()
    nu0 = np.r_[w.s('S_BOMEGA', 3), w.s('S_BVEL', 3), w.s('S_QD', nd)] if floating else w.s('S_QD', nd).copy()
    qdd = rng.uniform(-1, 1, n)
    tau = dynamics(sc, w.state, w.param, 0, qdd=qdd)[2]
    fb = n - nd
    w.s('S_JTORQUE', nd)[:] = tau[fb:]
    if floating:   # the base wrench as an external torque / force on the base (frame 0)
        w.s('S_EXTT', 3)[:] = tau[0:3]
        w.s('S_EXTF', 3)[:] = tau[3:6]
    w.step_physics()
    nu1 = np.r_[w.s('S_BOMEGA', 3), w.s('S_BVEL', 3), w.s('S_QD', nd)] if floating else w.s('S_QD', nd).copy()
    got = (nu1 - nu0) / dt
    assert np.abs(got - qdd).max() <= 1e-6 * np.abs(qdd).max()


# ---------------------------------------------------------------- (3) fp32 emulation vs the fp64 reference --------------
def _compare(env, rows, qdd_seed=5):
    """Every movable model: J of its last link at a point, M, tau at the state's nu and a random qdd, against the reference for the
    environments `rows`; 1e-5 of the environment's largest reference entry."""
    sc = env.scene
    st, pr = env.world.state.cpu().numpy(), env.world.param.cpu().numpy()
    checked = 0
    for m in _movable(env):
        n = n_coords(sc, m.uid)
        link = m.num_joints() - 1
        point = (0.03, -0.02, 0.01)
        g = torch.Generator().manual_seed(qdd_seed)
        qdd = torch.rand((env.num_envs, n), generator=g).mul_(2).sub_(1).to(env.world.state.device)
        Jl, Ja = m.jacobian(link, point)
        M, tau = m.mass_matrix(), m.inverse_dynamics(qdd=qdd)
        J = torch.cat([Jl, Ja], 1).cpu().numpy()
        M, tau, qdd = M.cpu().numpy(), tau.cpu().numpy(), qdd.cpu().numpy()
        for e in rows:
            Jr, Mr, tr = dynamics(sc, st[e], pr[e], m.uid, link, point, qdd=qdd[e])
            for got, ref, what in ((J[e], Jr, 'J'), (M[e], Mr, 'M'), (tau[e], tr, 'tau')):
                err = np.abs(got - ref).max()
                assert err <= 1e-5 * max(np.abs(ref).max(), 1e-30), (m.name, e, what, err, np.abs(ref).max())
        checked += 1
    assert checked > 0


def _random_steps(env, k, seed=0):
    g = torch.Generator(device=env.world.state.device).manual_seed(seed)
    for _ in range(k):
        env.step(env.sample_action(g))


@pytest.mark.parametrize('folder,name', SCENES)
def test_emulation_matches_reference(folder, name):
    env = _emul_env(folder, name, 4)
    _compare(env, range(4))
    _random_steps(env, 10)
    _compare(env, range(4))


# ---------------------------------------------------------------- (4) host layer on the emulated world -----------------
def test_shapes_columns_and_defaults():
    env = _emul_env('from_the_readme', 'from_the_readme', 3)
    _random_steps(env, 3)
    sc, N = env.scene, 3
    for m in _movable(env):
        n, nd = n_coords(sc, m.uid), m.body.n_dofs
        Jl, Ja = m.jacobian(m.num_joints() - 1, (0.1, 0, 0))
        assert Jl.shape == (N, 3, n) and Ja.shape == (N, 3, n)
        assert m.mass_matrix().shape == (N, n, n) and m.inverse_dynamics().shape == (N, n)
        # columns: a floating base's angular then linear velocity, then the DoF in movable_joints() order
        if m.body.kind == 2:
            assert torch.equal(m.jacobian(-1)[0][:, :, 3:6], torch.eye(3).expand(N, 3, 3))
            assert torch.equal(m.jacobian(-1)[1][:, :, 0:3], torch.eye(3).expand(N, 3, 3))
        q, qd, _ = m.joint_state()
        nu = qd if m.body.kind != 2 else torch.cat([m.base_velocity()[1], m.base_velocity()[0], qd], 1)
        # q=None / qd=None read the state row: bit for bit what passing the state's values gives
        assert torch.equal(m.mass_matrix(), m.mass_matrix(q.contiguous()))
        assert torch.equal(m.inverse_dynamics(), m.inverse_dynamics(q.contiguous(), nu.contiguous(), torch.zeros(N, n)))
        for a, b in zip(m.jacobian(0, (0.1, 0, 0)), m.jacobian(0, (0.1, 0, 0), q.contiguous())):
            assert torch.equal(a, b)
        assert q.shape[1] == nd


def test_validation_errors():
    env = _emul_env('from_the_readme', 'from_the_readme', 2)
    robot, r2d2, table = env.models['robot'], env.models['r2d2'], env.models['table']
    n = n_coords(env.scene, robot.uid)
    for bad in (lambda: table.mass_matrix(), lambda: env.models['plane'].inverse_dynamics()):
        with pytest.raises(ValueError):
            bad()
    with pytest.raises(ValueError):
        robot.mass_matrix(torch.zeros(2, n + 1))                       # wrong shape
    with pytest.raises(ValueError):
        robot.mass_matrix(torch.zeros(2, robot.body.n_dofs, dtype=torch.float64))   # wrong dtype
    with pytest.raises(ValueError):
        robot.inverse_dynamics(qd=torch.zeros(3, n))                  # wrong number of environments
    with pytest.raises(ValueError):
        robot.inverse_dynamics(qdd=torch.zeros(2, n, device='meta'))  # wrong device
    with pytest.raises(ValueError):
        r2d2.inverse_dynamics(qd=torch.zeros(2, r2d2.body.n_dofs))    # a floating base needs 6 more
    for f in (-2, robot.num_joints()):
        with pytest.raises(ValueError):
            robot.jacobian(f)
    fixed = [i for i in range(robot.num_joints()) if i not in robot.body.movable_joints()]
    for ids in ([fixed[0]], [robot.num_joints()], [-1]):
        with pytest.raises(ValueError):
            robot.apply_joint_torque(ids, 1.0)
        with pytest.raises(ValueError):
            robot.disable_motors(ids)
    with pytest.raises(ValueError):
        robot.apply_joint_torque(robot.body.movable_joints()[:2], torch.zeros(2, 3))
    with pytest.raises(ValueError):   # constructor-time only
        robot.disable_motors(robot.body.movable_joints()[:1])


def test_coordinate_limit():
    """A floating body with 60 revolute links (n = 66) is more than the kernel's 64 generalized coordinates."""
    import copy
    from diy_gym_b200.assets import resolve_model
    from diy_gym_b200.model import Model
    desc = copy.deepcopy(resolve_model('r2d2.urdf'))
    child = next(l for l in desc['links'][1:] if l['joint']['type'] in ('revolute', 'continuous'))
    desc['links'] = desc['links'][:1]
    for k in range(60):
        c = copy.deepcopy(child)
        c['name'], c['parent'] = 'l%d' % k, 0
        c['joint'] = dict(c['joint'], name='j%d' % k)
        desc['links'].append(c)

    class World:
        state = torch.zeros(2, 1)
    env = type('Env', (), {})()
    from diy_gym_b200.compiler.scene import SceneBuilder
    env.builder, env.world = SceneBuilder(), World()
    m = Model.__new__(Model)
    m.name, m.env = 'star', env
    m.body = env.builder.add_body('star', desc, xyz=(0, 0, 1))
    m.uid = m.body.index
    assert m.body.kind == 2 and m.body.n_dofs == 60
    with pytest.raises(ValueError, match='at most 64'):
        m.mass_matrix()


def test_disable_motors_in_constructor_and_joint_torque_cleared_by_step(tmp_path):
    class MotorsOff(Addon):
        def __init__(self, parent, config):
            super().__init__(parent, config)
            self.ids = parent.body.movable_joints()[1:3]
            parent.disable_motors(self.ids)
    AddonFactory.register_addon('test_motors_off', MotorsOff)
    path = tmp_path / 'motors_off.yaml'
    path.write_text('ur5:\n  model: ur5/ur5_robot.urdf\n  off: {addon: test_motors_off}\n')
    env = _emul_env(None, None, 2, str(path))
    ur5, sc = env.models['ur5'], env.scene
    dofs = [ur5.body.global_dof(i) for i in ur5.body.movable_joints()]
    mmaxf = sc.sec['STATE_DEFAULT'][sc.hdr['S_MMAXF'] + np.array(dofs)]
    assert np.array_equal(mmaxf == 0, np.isin(np.arange(len(dofs)), [1, 2]))
    assert (env.world.state[:, sc.hdr['S_MMAXF'] + torch.tensor(dofs)][:, [1, 2]] == 0).all()
    ids = ur5.body.movable_joints()[:2]
    ur5.apply_joint_torque(ids, torch.tensor([[1., 2.], [3., 4.]]))
    ur5.apply_joint_torque(ids, 0.5)
    jt = env.world.state[:, sc.hdr['S_JTORQUE'] + torch.tensor(dofs[:2])]
    assert torch.equal(jt, torch.tensor([[1.5, 2.5], [3.5, 4.5]]))
    env.world.step()
    assert (env.world.state[:, sc.hdr['S_JTORQUE']:sc.hdr['S_JTORQUE'] + sc['nd']] == 0).all()


# ---------------------------------------------------------------- (5) admittance_controller as a user add-on -------------
class UserAdmittance(Addon):
    """admittance_controller.py of the reference on the dynamics queries: tau = J_lin^T F + J_ang^T T + inverse_dynamics(q, 0, 0)
    + kp (target - q) - kd qd, applied as joint torques, default motors off."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.model = parent
        self.end_frame = parent.get_frame_id(config.get('end_effector'))
        self.offset = list(config.get('offset_admittance_point', [0., 0., 0.]))
        self.kp, self.kd = config.get('p_gain', 0.001), config.get('d_gain', 0.01)
        self.joint_ids = [i for i in parent.body.movable_joints() if i <= self.end_frame]
        rest = config.get('rest_position', [0.] * len(self.joint_ids))
        self.target = torch.tensor(config.get('target_pose', rest), dtype=torch.float32)
        parent.disable_motors(self.joint_ids)
        self.action_space = spaces.Dict({'force': spaces.Box(-5, 5, shape=(3, ), dtype='float32'),
                                         'torque': spaces.Box(-1., 1., shape=(3, ), dtype='float32')})

    def update(self, action):
        m = self.model
        q, qd, _ = m.joint_state(self.joint_ids)
        Jl, Ja = m.jacobian(self.end_frame, self.offset)
        F, T = action['force'], action['torque']
        g = m.inverse_dynamics(q.contiguous(), torch.zeros_like(q))
        tau = (Jl.transpose(1, 2) @ F[..., None])[..., 0] + (Ja.transpose(1, 2) @ T[..., None])[..., 0] + g
        m.apply_joint_torque(self.joint_ids, tau + self.kp * (self.target.to(q.device) - q) - self.kd * qd)


def _admittance_parity(tmp_path, factory, n):
    AddonFactory.register_addon('user_admittance', UserAdmittance)
    src = os.path.join(EX, 'ur_admittance', 'ur_admittance.yaml')
    path = tmp_path / 'ur_admittance_user.yaml'
    with open(src) as f:
        path.write_text(f.read().replace('addon: admittance_controller', 'addon: user_admittance'))
    a = _env('ur_admittance', 'ur_admittance', n, factory)
    b = _env(None, None, n, factory, str(path))
    ha, hb = a.scene.hdr, b.scene.hdr
    assert all(ha[k] == hb[k] for k in ha if k.startswith('S_') or k == 'S')
    ka = a.scene.sec['STATE_DEFAULT'][ha['S_MMAXF']:ha['S_MMAXF'] + a.scene['nd']]
    assert np.array_equal(ka, b.scene.sec['STATE_DEFAULT'][hb['S_MMAXF']:hb['S_MMAXF'] + b.scene['nd']])
    g = torch.Generator(device=a.world.state.device).manual_seed(7)
    _random_steps(a, 5, seed=1)
    nd = a.scene['nd']
    q0 = ha['S_Q']
    for _ in range(10):
        b.world.state.copy_(a.world.state)
        b.world.param.copy_(a.world.param)
        act = a.sample_action(g)
        a.step(act)
        b.step(act)
        qa, qb = a.world.state[:, q0:q0 + nd].cpu().double(), b.world.state[:, q0:q0 + nd].cpu().double()
        da, db = a.world.state[:, ha['S_QD']:ha['S_QD'] + nd].cpu().double(), b.world.state[:, hb['S_QD']:hb['S_QD'] + nd].cpu().double()
        assert (qa - qb).abs().max() <= 1e-4 * qa.abs().max()
        assert (da - db).abs().max() <= 1e-4 * max(da.abs().max().item(), 1e-2)
    return a, b


def test_admittance_controller_as_user_addon(tmp_path):
    from tests.emul.dyn_emul import factory
    _admittance_parity(tmp_path, factory(4), 4)


# ---------------------------------------------------------------- GPU ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('folder,name', SCENES)
def test_kernel_matches_reference_gpu(folder, name):
    env = _env(folder, name, 4096)
    _random_steps(env, 10)
    rows = np.random.default_rng(0).choice(4096, 64, replace=False)
    _compare(env, sorted(rows.tolist()) + [4095])
    env.close()
    env = _env(folder, name, 37)   # a partial last block of four environments
    _random_steps(env, 3)
    _compare(env, range(37))
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('folder,name', [('r2d2_maze', 'r2d2_maze'), ('from_the_readme', 'from_the_readme')])
def test_jacobian_times_velocity_equals_link_cache_gpu(folder, name):
    env = _env(folder, name, 512)
    _random_steps(env, 20)
    h, st = env.scene.hdr, env.world.state
    for m in _movable(env):
        b = m.body
        nu = st[:, h['S_QD'] + b.dof_start:h['S_QD'] + b.dof_start + b.n_dofs]
        if b.kind == 2:
            v, om = m.base_velocity()
            nu = torch.cat([om, v, nu], 1)
        vl = st[:, h['S_LVEL'] + 3 * b.link_start:h['S_LVEL'] + 3 * (b.link_start + b.n_links)].reshape(-1, b.n_links, 3)
        wl = st[:, h['S_LOMEGA'] + 3 * b.link_start:h['S_LOMEGA'] + 3 * (b.link_start + b.n_links)].reshape(-1, b.n_links, 3)
        scale = torch.clamp(torch.cat([vl, wl], 1).norm(dim=2).max(dim=1).values, min=1e-2)
        for k in range(b.n_links):
            Jl, Ja = m.jacobian(k)
            ev = ((Jl @ nu[..., None])[..., 0] - vl[:, k]).abs().max(dim=1).values
            ew = ((Ja @ nu[..., None])[..., 0] - wl[:, k]).abs().max(dim=1).values
            assert (ev <= 1e-5 * scale).all() and (ew <= 1e-5 * scale).all(), (m.name, k, float(ev.max()), float(ew.max()))
    env.close()


@pytest.mark.gpu
def test_no_side_effects_streams_and_explicit_state_gpu():
    env = _env('from_the_readme', 'from_the_readme', 256)
    _random_steps(env, 5)
    w = env.world
    before = [t.clone() for t in (w.state, w.param, w.obs, w.reward, w.term)]

    def all_queries(m, **kw):
        n = n_coords(env.scene, m.uid)
        qdd = torch.linspace(-1, 1, n, device='cuda').expand(256, n).contiguous()
        return list(m.jacobian(m.num_joints() - 1, (0.01, 0.02, 0.03), **kw)) + [m.mass_matrix(**kw), m.inverse_dynamics(qdd=qdd, **kw)]
    models = _movable(env)
    ref = [all_queries(m) for m in models]
    torch.cuda.synchronize()
    for a, b in zip(before, (w.state, w.param, w.obs, w.reward, w.term)):
        assert torch.equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = [all_queries(m) for m in models]
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for r, g in zip(ref, got):
        assert all(torch.equal(x, y) for x, y in zip(r, g))
    for m, r in zip(models, ref):
        q = m.joint_state()[0].contiguous()
        assert all(torch.equal(x, y) for x, y in zip(r, all_queries(m, q=q)))
    env.close()


@pytest.mark.gpu
def test_admittance_controller_as_user_addon_gpu(tmp_path):
    a, b = _admittance_parity(tmp_path, None, 64)
    a.close()
    b.close()
