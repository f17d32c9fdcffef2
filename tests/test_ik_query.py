"""Batched inverse kinematics of a Model (pybullet's calculateInverseKinematics: csrc/dg_ik.cuh + dg_ik_kernel over the step
kernel's ik_solve*) and position-motor targets (setJointMotorControlArray(POSITION_CONTROL)).

CPU: the fp64 reference (tests/ik_reference.py) is pinned to the oracle's IK; the g++ build of dg_ik.cuh (tests/emul)
is checked against it on every template path; known answers; the host layer and its errors on the emulated world; the
reference's ik_controller written as a user add-on on these calls; set_position_targets against joint_controller.  GPU: the same
checks on the kernel, plus side effects and streams."""
import copy
import math
import os
import tempfile

import numpy as np
import pytest
import torch

from diy_gym_b200 import spaces
from diy_gym_b200 import torch_math as tm
from diy_gym_b200.addons.addon import Addon, AddonFactory
from diy_gym_b200.compiler.mathutil import quat_from_euler, quat_mul
from oracle.oracle import OracleWorld
from tests.helpers import build_single
from tests.ik_reference import fk, ik

EX = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'examples')
# (folder, yaml): UR5 (6 DoF: ik_solve_fast<6, M>), Jaco (10 DoF) and floating R2D2 (8 DoF): <12, M>; a UR5 with the
# three-finger gripper (17 DoF, GENERIC below): the generic ik_solve
SCENES = [('ur_high_5', 'ur_high_5'), ('from_the_readme', 'from_the_readme'), ('r2d2_maze', 'r2d2_maze'), (None, 'ur5_3f')]
GENERIC = {'ur5_3f': 'arm:\n  model: ur5/ur5_3f.urdf\n  xyz: [0.1, -0.2, 0.3]\n  rpy: [0.0, 0.0, 0.5]\n'}


def _env(folder, name, n, factory=None, path=None):
    from bench import register_example_addons
    from diy_gym_b200 import DIYGym
    register_example_addons()
    if path is None and folder is None:
        path = os.path.join(tempfile.mkdtemp(), name + '.yaml')
        with open(path, 'w') as f:
            f.write(GENERIC[name])
    return DIYGym(path or os.path.join(EX, folder, name + '.yaml'), num_envs=n, device=0, seed=4321, world_factory=factory)


def _emul_factory(team=4):
    from tests.emul.world import factory
    return factory(team)


def _emul_env(folder, name, n=4, path=None):
    return _env(folder, name, n, _emul_factory(), path)


def _models(receptor):
    for m in receptor.models.values():
        yield m
        yield from _models(m)


def _movable(env):
    return [m for m in _models(env) if m.body.n_dofs > 0]


def _random_steps(env, k, seed=0):
    g = torch.Generator(device=env.world.state.device).manual_seed(seed)
    for _ in range(k):
        env.step(env.sample_action(g))


def _deepest_link(body):
    """The link with the most movable joints between it and the base (the last of those on a tie)."""
    best, nbest = 0, -1
    for j in range(body.num_joints()):
        k, n = j + 1, 0
        while k > 0:
            n += body.links[k]['joint']['type'] != 'fixed'
            k = body.links[k]['parent']
        if n >= nbest:
            best, nbest = j, n
    return best


def _f32(x, dev):
    return torch.as_tensor(np.asarray(x), dtype=torch.float32, device=dev).contiguous()


def _problem(env, m, seed, spread=0.3):
    """Targets from FK of the state's q plus a random offset, and synthetic null-space lists: every seed is inside [lower, upper]
    except on every third joint, where it lies above `upper` so that the limit term acts."""
    sc, st = env.scene, env.world.state.cpu().numpy().astype(np.float64)
    b, link, N = m.body, _deepest_link(m.body), env.num_envs
    rng = np.random.default_rng(seed)
    q = st[:, sc.hdr['S_Q'] + b.dof_start:sc.hdr['S_Q'] + b.dof_start + b.n_dofs]
    qs = q + rng.uniform(-spread, spread, q.shape)
    poses = [fk(sc, st[e], m.uid, link, qs[e]) for e in range(N)]
    tpos, torn = np.array([p for p, _ in poses]), np.array([o for _, o in poses])
    lower = q - 1.0
    upper = q + np.where(np.arange(b.n_dofs) % 3 == 2, -0.05, 1.0)
    lims = np.stack([lower, upper, upper - lower, q + 0.1], 1)
    return link, tpos, torn, lims


def _check_against_reference(env, rows, seed=0, iters=20, qtol=1e-4, etol=1e-5):
    """Every movable model, position and pose targets, with and without the null-space lists, threshold 0 (so that the early
    exit cannot differ between fp32 and fp64): q and err against the reference, rows `rows`.  Returns the largest deviations."""
    sc, dev = env.scene, env.world.state.device
    st = env.world.state.cpu().numpy()
    worst = [0.0, 0.0]
    paths = set()
    for m in _movable(env):
        link, tpos, torn, lims = _problem(env, m, seed)
        for use_orn in (False, True):
            for ns in (False, True):
                kw = dict(zip(('lower_limits', 'upper_limits', 'joint_ranges', 'rest_poses'), [_f32(lims[:, i], dev) for i in range(4)])) if ns else {}
                q, err = m.inverse_kinematics(link, _f32(tpos, dev), _f32(torn, dev) if use_orn else None, max_iterations=iters,
                                              residual_threshold=0.0, return_error=True, **kw)
                q, err = q.cpu().numpy(), err.cpu().numpy()
                for e in rows:
                    qr, er = ik(sc, st[e], m.uid, link, tpos[e], torn[e] if use_orn else None, None, tuple(lims[e]) if ns else None,
                                iters=iters, threshold=0.0)
                    dq, de = np.abs(q[e] - qr).max(), np.abs(err[e] - er).max()
                    assert dq <= qtol and de <= etol, (m.name, e, use_orn, ns, dq, de)
                    worst = [max(worst[0], dq), max(worst[1], de)]
                paths.add((6 if m.body.n_dofs <= 6 else 12 if m.body.n_dofs <= 12 else 0, use_orn, ns, m.body.kind == 2))
    return worst, paths


# ---------------------------------------------------------------- (1) the reference, pinned to the oracle --------------
LIMB = [('ur5/ur5_robot.urdf', True, 'ee_fixed_joint'), ('jaco/j2s7s300_standalone.urdf', True, 'j2s7s300_joint_end_effector'),
        ('r2d2.urdf', False, 'left_tip_joint')]


@pytest.mark.parametrize('model,fixed,frame', LIMB)
@pytest.mark.parametrize('use_orn', [False, True])
@pytest.mark.parametrize('nullspace', [False, True])
def test_reference_equals_oracle_ik(model, fixed, frame, use_orn, nullspace):
    sc = build_single(model, fixed_base=fixed, xyz=(0.3, 0.1, 0.5), quat=quat_from_euler([0.1, -0.2, 0.7]))
    w = OracleWorld(sc)
    b, nd = sc.bodies[0], sc['nd']
    link = b.joint_index(frame)
    rng = np.random.default_rng(0)
    q0 = rng.uniform(-0.5, 0.5, nd)
    w.s('S_Q', nd)[:] = q0
    w.refresh()
    p, o = fk(sc, w.state, 0, link, q0)
    tpos, torn = p + [0.03, -0.02, 0.04], quat_mul(o, quat_from_euler([0.05, 0.02, -0.03]))
    infos = [b.joint_info(i) for i in b.movable_joints()]
    lo, up = np.array([i['lower'] for i in infos]), np.array([i['upper'] for i in infos])
    lims = (lo, up, up - lo, rng.uniform(-1, 1, nd)) if nullspace else None
    want = w.ik(0, b.link_start + link, tpos, torn if use_orn else None, lims)
    got, err = ik(sc, w.state, 0, link, tpos, torn if use_orn else None, limits=lims)
    assert np.abs(got - want).max() <= 1e-9
    # err is the residual at the returned q
    p1, o1 = fk(sc, w.state, 0, link, got)
    assert abs(err[0] - np.linalg.norm(tpos - p1)) <= 1e-12
    if not use_orn:
        assert err[1] == 0


# ---------------------------------------------------------------- (2) fp32 emulation vs the fp64 reference --------------
@pytest.mark.parametrize('folder,name', SCENES)
def test_emulation_matches_reference(folder, name):
    env = _emul_env(folder, name, 4)
    _random_steps(env, 5)
    worst, paths = _check_against_reference(env, range(4))
    print('%s: max |dq| %.2e rad, max |d err| %.2e' % (name, *worst))


def test_emulation_covers_every_template_path():
    paths = set()
    for folder, name in SCENES:
        env = _emul_env(folder, name, 2)
        paths |= _check_against_reference(env, range(2))[1]
    for maxd in (6, 12, 0):
        for use_orn in (False, True):
            assert (maxd, use_orn, False, False) in paths or (maxd, use_orn, False, True) in paths, (maxd, use_orn)
            assert (maxd, use_orn, True, False) in paths or (maxd, use_orn, True, True) in paths, (maxd, use_orn)
    assert (12, True, True, True) in paths and (12, False, True, True) in paths   # null-space on a floating base (R2D2)


# ---------------------------------------------------------------- (3) known answers -------------------------------------
@pytest.mark.parametrize('folder,name,use_orn', [('ur_high_5', 'ur_high_5', True), ('from_the_readme', 'from_the_readme', False)])
def test_known_answers_converge(folder, name, use_orn):
    """target = FK(q*) for q* inside the limits, seed q* + delta (|delta| <= 0.1 rad), 200 iterations: wherever the reference
    reaches 1e-4 m, the query's own err is within 1e-3 m."""
    env = _emul_env(folder, name, 8)
    _check_known_answers(env, use_orn)


def _check_known_answers(env, use_orn, rows=None):
    sc, dev, N = env.scene, env.world.state.device, env.num_envs
    st = env.world.state.cpu().numpy()
    rng = np.random.default_rng(11)
    reached = 0
    for m in _movable(env):
        if m.body.kind == 2:
            continue
        b, link = m.body, _deepest_link(m.body)
        infos = [b.joint_info(i) for i in b.movable_joints()]
        lo = np.array([i['lower'] if i['lower'] < i['upper'] else -np.pi for i in infos])
        up = np.array([i['upper'] if i['lower'] < i['upper'] else np.pi for i in infos])
        qs = rng.uniform(lo + 0.1 * (up - lo), up - 0.1 * (up - lo), (N, b.n_dofs))
        seed = qs + rng.uniform(-0.1, 0.1, qs.shape)
        poses = [fk(sc, st[e], m.uid, link, qs[e]) for e in range(N)]
        tpos, torn = np.array([p for p, _ in poses]), np.array([o for _, o in poses])
        q, err = m.inverse_kinematics(link, _f32(tpos, dev), _f32(torn, dev) if use_orn else None, q=_f32(seed, dev),
                                      max_iterations=200, return_error=True)
        err = err.cpu().numpy()
        for e in (range(N) if rows is None else rows):
            _, er = ik(sc, st[e], m.uid, link, tpos[e], torn[e] if use_orn else None, seed[e], iters=200)
            if er[0] <= 1e-4:
                reached += 1
                assert err[e, 0] <= 1e-3, (m.name, e, err[e], er)
    assert reached > 0


def test_seed_default_and_quaternion_norm():
    env = _emul_env('ur_high_5', 'ur_high_5', 4)
    _random_steps(env, 3)
    m = env.models['ur5_l']
    link, tpos, torn, _ = _problem(env, m, 3)
    tpos, torn = _f32(tpos, 'cpu'), _f32(torn, 'cpu')
    q, err = m.inverse_kinematics(link, tpos, torn, return_error=True)
    q2, err2 = m.inverse_kinematics(link, tpos, torn, q=m.joint_state()[0].contiguous(), return_error=True)
    assert torch.equal(q, q2) and torch.equal(err, err2)
    # a power-of-two scale normalises to the same bits; any other norm to the same rotation
    q3, err3 = m.inverse_kinematics(link, tpos, 2.0 * torn, return_error=True)
    assert torch.equal(q, q3) and torch.equal(err, err3)
    qa, ea = m.inverse_kinematics(link, tpos, torn, residual_threshold=0.0, return_error=True)
    qb, eb = m.inverse_kinematics(link, tpos, 0.37 * torn, residual_threshold=0.0, return_error=True)
    assert (qa - qb).abs().max() <= 1e-5 and (ea - eb).abs().max() <= 1e-5


# ---------------------------------------------------------------- (4) host layer -----------------------------------------
def test_shapes_broadcasting_and_no_side_effects():
    env = _emul_env('from_the_readme', 'from_the_readme', 3)
    _random_steps(env, 2)
    w, N = env.world, 3
    before = [t.clone() for t in (w.state, w.param, w.obs, w.reward, w.term)]
    for m in _movable(env):
        nd, link = m.body.n_dofs, _deepest_link(m.body)
        p = torch.tensor([0.1, 0.5, 0.9])
        o = torch.tensor([0.0, 0.0, 0.38268343, 0.92387953])
        q = m.inverse_kinematics(link, p)
        assert q.shape == (N, nd) and q.dtype == torch.float32
        q1, err = m.inverse_kinematics(link, p.expand(N, 3).contiguous(), o.expand(N, 4).contiguous(), return_error=True)
        assert err.shape == (N, 2) and torch.equal(q1, m.inverse_kinematics(link, p, o))
        assert torch.equal(q, m.inverse_kinematics(link, p.expand(N, 3).contiguous()))
        lists = [torch.zeros(nd) - 1, torch.zeros(nd) + 1, torch.zeros(nd) + 2, torch.zeros(nd)]
        a = m.inverse_kinematics(link, p, None, None, *lists)
        b = m.inverse_kinematics(link, p, None, None, *[t.expand(N, nd).contiguous() for t in lists])
        assert torch.equal(a, b) and not torch.equal(a, q)
    for a, b in zip(before, (w.state, w.param, w.obs, w.reward, w.term)):
        assert torch.equal(a, b)


def test_validation_errors():
    env = _emul_env('from_the_readme', 'from_the_readme', 2)
    robot, table = env.models['robot'], env.models['table']
    nd, p = robot.body.n_dofs, torch.zeros(3)
    ik = robot.inverse_kinematics
    bad = [lambda: ik(-1, p), lambda: ik(robot.num_joints(), p), lambda: table.inverse_kinematics(0, p),
           lambda: ik(3, torch.zeros(3, dtype=torch.float64)), lambda: ik(3, [0., 0., 0.]), lambda: ik(3, torch.zeros(3, 3)),
           lambda: ik(3, torch.zeros(2, 3, device='meta')), lambda: ik(3, p, torch.zeros(3)), lambda: ik(3, p, q=torch.zeros(nd)),
           lambda: ik(3, p, q=torch.zeros(2, nd + 1)), lambda: ik(3, p, lower_limits=torch.zeros(nd)),
           lambda: ik(3, p, None, None, torch.zeros(nd), torch.zeros(nd), torch.zeros(nd)),
           lambda: ik(3, p, None, None, *[torch.zeros(nd - 1)] * 4), lambda: ik(3, p, max_iterations=0),
           lambda: ik(3, p, max_iterations=2.5), lambda: ik(3, p, residual_threshold=-1.0), lambda: ik(3, p, residual_threshold=math.nan)]
    for k, f in enumerate(bad):
        with pytest.raises(ValueError):
            f()
            print(k)
    fixed = [i for i in range(robot.num_joints()) if i not in robot.body.movable_joints()]
    for ids in ([fixed[0]], [robot.num_joints()], [-1]):
        with pytest.raises(ValueError):
            robot.set_position_targets(ids, 0.0)
    with pytest.raises(ValueError):
        robot.set_position_targets(robot.body.movable_joints()[:2], torch.zeros(2, 3))
    with pytest.raises(ValueError):
        robot.set_position_targets(robot.body.movable_joints()[:2], 0.0, max_force=torch.zeros(3))


def test_dof_limit():
    """A body with 70 revolute links is more than the query's 64 DoF."""
    from diy_gym_b200.assets import resolve_model
    from diy_gym_b200.compiler.scene import SceneBuilder
    from diy_gym_b200.model import Model
    desc = copy.deepcopy(resolve_model('r2d2.urdf'))
    child = next(l for l in desc['links'][1:] if l['joint']['type'] in ('revolute', 'continuous'))
    desc['links'] = desc['links'][:1]
    for k in range(70):
        c = copy.deepcopy(child)
        c['name'], c['parent'] = 'l%d' % k, 0
        c['joint'] = dict(c['joint'], name='j%d' % k)
        desc['links'].append(c)

    class World:
        state = torch.zeros(2, 1)
    env = type('Env', (), {})()
    env.builder, env.world = SceneBuilder(), World()
    m = Model.__new__(Model)
    m.name, m.env = 'star', env
    m.body = env.builder.add_body('star', desc, xyz=(0, 0, 1))
    m.uid = m.body.index
    with pytest.raises(ValueError, match='at most 64'):
        m.inverse_kinematics(0, torch.zeros(3))


# ---------------------------------------------------------------- (5) ik_controller as a user add-on ---------------------
class UserIK(Addon):
    """ik_controller.py of the reference on the query: target = COM pose of the end effector + the action's delta (orientation
    quat * euler(delta)), inverse_kinematics (with the four null-space lists exactly when the built-in op uses them), position
    targets on the arm's joints with gains 0.015 / 1.0."""
    resets_in_constructor = True

    def __init__(self, parent, config):
        super().__init__(parent, config)
        b = parent.body
        self.model = parent
        self.ee = b.joint_names().index(config.get('end_effector'))
        self.joint_ids = [i for i in b.movable_joints() if i <= self.ee]
        self.rest_position = list(config.get('rest_position', [0] * len(self.joint_ids)))
        self.use_orientation = bool(config.get('use_orientation', False))
        self.lists = None
        if len(self.joint_ids) == b.n_dofs and len(self.rest_position) == b.n_dofs:
            infos = [b.joint_info(i) for i in self.joint_ids]
            lo, up = [i['lower'] for i in infos], [i['upper'] for i in infos]
            self.lists = [torch.tensor(v, dtype=torch.float32) for v in (lo, up, [u - l for l, u in zip(lo, up)], self.rest_position)]
        self.action_space = spaces.Dict({'linear': spaces.Box(-0.01, 0.01, shape=(3, ), dtype='float32')})
        if self.use_orientation:
            self.action_space.spaces['rotation'] = spaces.Box(-0.01, 0.01, shape=(3, ), dtype='float32')

    def update(self, action):
        m = self.model
        pos, quat = m.link_state(self.ee)[:2]
        dev = pos.device
        tpos = (pos + action['linear'].to(dev)).contiguous()
        torn = tm.quat_mul(quat, tm.quat_from_euler(action['rotation'].to(dev))).contiguous() if self.use_orientation else None
        kw = {}
        if self.lists is not None:
            kw = dict(zip(('lower_limits', 'upper_limits', 'joint_ranges', 'rest_poses'), [t.to(dev) for t in self.lists]))
        q = m.inverse_kinematics(self.ee, tpos, torn, **kw)
        m.set_position_targets(self.joint_ids, q[:, :len(self.joint_ids)], 0.015, 1.0)


def _user_scene(tmp_path, folder, name, old, new):
    path = tmp_path / ('%s_user.yaml' % name)
    with open(os.path.join(EX, folder, name + '.yaml')) as f:
        text = f.read()
    assert old in text
    path.write_text(text.replace(old, new))
    return str(path)


def _ik_parity(tmp_path, folder, name, factory, n, strict):
    AddonFactory.register_addon('user_ik', UserIK)
    a = _env(folder, name, n, factory)
    b = _env(None, None, n, factory, _user_scene(tmp_path, folder, name, 'addon: ik_controller', 'addon: user_ik'))
    ha, hb = a.scene.hdr, b.scene.hdr
    assert all(ha[k] == hb[k] for k in ha if k.startswith('S_') or k == 'S')
    dofs = [d for m in _models(a) for ad in m.addons.values() if type(ad).__name__ == 'InverseKinematicsController'
            for d in (m.body.global_dof(i) for i in ad.joint_ids)]
    assert dofs
    cols = torch.tensor(dofs) + ha['S_MTPOS']
    nd, q0, qd0 = a.scene['nd'], ha['S_Q'], ha['S_QD']
    g = torch.Generator(device=a.world.state.device).manual_seed(7)
    _random_steps(a, 5, seed=1)
    worst = 0.0
    for _ in range(10):
        b.world.state.copy_(a.world.state)
        b.world.param.copy_(a.world.param)
        act = a.sample_action(g)
        a.step(act)
        b.step(act)
        ta, tb = a.world.state[:, cols.to(a.world.state.device)].cpu(), b.world.state[:, cols.to(b.world.state.device)].cpu()
        worst = max(worst, (ta - tb).abs().max().item())
        assert worst <= 1e-4, worst
        if strict:
            qa, qb = a.world.state[:, q0:q0 + nd].cpu().double(), b.world.state[:, q0:q0 + nd].cpu().double()
            da, db = a.world.state[:, qd0:qd0 + nd].cpu().double(), b.world.state[:, qd0:qd0 + nd].cpu().double()
            assert (qa - qb).abs().max() <= 1e-4 * qa.abs().max()
            assert (da - db).abs().max() <= 1e-4 * max(da.abs().max().item(), 1e-2)
    print('%s: max |S_MTPOS difference| over 10 steps %.3e rad' % (name, worst))
    return a, b


IK_SCENES = [('ur_high_5', 'ur_high_5', True), ('ur_gripper', 'ur_gripper', False), ('from_the_readme', 'from_the_readme', False)]


@pytest.mark.parametrize('folder,name,strict', IK_SCENES)
def test_ik_controller_as_user_addon(tmp_path, folder, name, strict):
    _ik_parity(tmp_path, folder, name, _emul_factory(8), 4, strict)   # (the welded payload of ur_gripper needs a team of 8)


# ---------------------------------------------------------------- (6) set_position_targets = joint_controller ------------
class UserPositionTargets(Addon):
    """joint_controller in position mode on the motor call: every movable joint, gains 0.03 / 1.0, the URDF effort."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.model = parent
        self.joint_ids = parent.body.movable_joints()
        self.action_space = spaces.Box(-0.5, 0.5, shape=(len(self.joint_ids), ), dtype='float32')

    def update(self, action):
        self.model.set_position_targets(self.joint_ids, action.to(self.model.world.state.device), 0.03, 1.0)


POSITION_YAML = 'ur5:\n  model: ur5/ur5_robot.urdf\n  controller: {addon: %s}\n'


def _position_parity(tmp_path, factory, n):
    AddonFactory.register_addon('user_position_targets', UserPositionTargets)
    pa, pb = tmp_path / 'joint_position.yaml', tmp_path / 'user_position.yaml'
    pa.write_text(POSITION_YAML % 'joint_controller, control_mode: position')
    pb.write_text(POSITION_YAML % 'user_position_targets')
    a, b = _env(None, None, n, factory, str(pa)), _env(None, None, n, factory, str(pb))
    assert all(a.scene.hdr[k] == b.scene.hdr[k] for k in a.scene.hdr if k.startswith('S_') or k == 'S')
    cfg = lambda w: tuple(getattr(w, k, None) for k in ('team', 'block_threads', 'grid_blocks', 'smem_bytes'))
    same_launch = cfg(a.world) == cfg(b.world)
    g = torch.Generator(device=a.world.state.device).manual_seed(3)
    _random_steps(a, 3, seed=2)
    nd, h = a.scene['nd'], a.scene.hdr
    for _ in range(3):
        b.world.state.copy_(a.world.state)
        b.world.param.copy_(a.world.param)
        act = a.sample_action(g)
        a.step(act)
        b.step(act)
        if same_launch:
            assert torch.equal(a.world.state, b.world.state)
        else:
            for o in (h['S_Q'], h['S_QD']):
                x, y = a.world.state[:, o:o + nd].cpu().double(), b.world.state[:, o:o + nd].cpu().double()
                assert (x - y).abs().max() <= 1e-4 * max(x.abs().max().item(), 1e-2)
    print('set_position_targets vs joint_controller: %s' % ('bit for bit' if same_launch else 'strict bar (launch configurations differ)'))
    return a, b


def test_set_position_targets_equals_joint_controller(tmp_path):
    _position_parity(tmp_path, _emul_factory(), 4)


# ---------------------------------------------------------------- GPU ------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('folder,name', SCENES)
def test_kernel_matches_reference_gpu(folder, name):
    env = _env(folder, name, 4096)
    _random_steps(env, 5)
    rows = sorted(np.random.default_rng(0).choice(4095, 24, replace=False).tolist()) + [4095]
    worst, _ = _check_against_reference(env, rows)
    print('%s 4096: max |dq| %.2e rad, max |d err| %.2e' % (name, *worst))
    env.close()
    env = _env(folder, name, 37)   # a partial block of 64 lanes
    _random_steps(env, 3)
    worst, _ = _check_against_reference(env, list(range(0, 36, 3)) + [36])
    print('%s 37: max |dq| %.2e rad, max |d err| %.2e' % (name, *worst))
    env.close()


@pytest.mark.gpu
def test_known_answers_gpu():
    env = _env('ur_high_5', 'ur_high_5', 1024)
    _check_known_answers(env, True, rows=range(0, 1024, 16))
    env.close()


@pytest.mark.gpu
def test_no_side_effects_streams_and_explicit_seed_gpu():
    env = _env('from_the_readme', 'from_the_readme', 256)
    _random_steps(env, 5)
    w = env.world
    before = [t.clone() for t in (w.state, w.param, w.obs, w.reward, w.term)]
    cases = []
    for m in _movable(env):
        link, tpos, torn, lims = _problem(env, m, 5)
        lists = [_f32(lims[:, i], 'cuda') for i in range(4)]
        cases.append((m, link, _f32(tpos, 'cuda'), _f32(torn, 'cuda'), lists))

    def run(**kw):
        return [m.inverse_kinematics(link, p, o, None, *lists, return_error=True, **kw) + m.inverse_kinematics(link, p, return_error=True, **kw)
                for m, link, p, o, lists in cases]
    ref = run()
    torch.cuda.synchronize()
    for a, b in zip(before, (w.state, w.param, w.obs, w.reward, w.term)):
        assert torch.equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = run()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for r, g in zip(ref, got):
        assert all(torch.equal(x, y) for x, y in zip(r, g))
    for (m, link, p, o, lists), r in zip(cases, ref):
        q = m.joint_state()[0].contiguous()
        got = m.inverse_kinematics(link, p, o, q, *lists, return_error=True) + m.inverse_kinematics(link, p, q=q, return_error=True)
        assert all(torch.equal(x, y) for x, y in zip(r, got))
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('folder,name,strict', IK_SCENES)
def test_ik_controller_as_user_addon_gpu(tmp_path, folder, name, strict):
    a, b = _ik_parity(tmp_path, folder, name, None, 64, strict)
    a.close()
    b.close()


@pytest.mark.gpu
def test_set_position_targets_equals_joint_controller_gpu(tmp_path):
    a, b = _position_parity(tmp_path, None, 64)
    a.close()
    b.close()
