"""ray_sensor add-on: host layer (pattern, spaces, validation), known answers of the fp64 reference (tests/ray_reference.py), the
fp32 device routines (g++ build, tests/emul/ray_emul.py) against it, and on the GPU the CUDA kernel through the C ABI against it and
against itself across schedules.  The oracle world (oracle/) is used for what it already offers: forward kinematics into the link
cache of a state row, and the step physics of the emulated legs."""
import os

import numpy as np
import pytest
import torch
import yaml

from diy_gym_b200.assets import resolve_model
from diy_gym_b200.compiler.mathutil import mat_to_quat, quat_to_mat
from diy_gym_b200.compiler.scene import KERNEL_OPS, OP, SceneBuilder, emit_c_header
from diy_gym_b200.config import Configuration
from diy_gym_b200.diy_gym import DIYGym
from diy_gym_b200.addons.builtin import RaySensor
from oracle.oracle import OracleWorld
from tests import ray_reference
from tests.emul.emul import EmulWorld
from tests.emul.ray_emul import RayCaster
from tools.ray_probe import maze_with_lidar, ray_ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# The maze's R2D2 spawns on the wall grid: from there ray 8 of 64 (45 degrees) runs exactly into the corner where two walls meet, a
# tie between two bodies that fp32 and fp64 break differently.  The parity legs turn the lidar by 0.7 degrees to keep clear of it.
MAZE_LIDAR = dict(include_hit_object=True, rpy=[0, 0, 0.0123])
EXAMPLE = os.path.join(ROOT, 'examples', 'ray_sensor', 'ray_sensor.yaml')


def example_config(**edit):
    with open(EXAMPLE) as f:
        node = yaml.load(f, Loader=yaml.FullLoader)
    for k, v in edit.items():
        node['r2d2']['lidar'][k] = v
    return node


def compile_config(node, name='ray_sensor'):
    return DIYGym(Configuration.from_dict(name, node), num_envs=1, compile_only=True)


# ---------------------------------------------------------------- host layer ----------------------------------------
def test_pattern_full_turn_and_fov_layer_major():
    d = RaySensor.pattern(4, 360.0, [0.0])
    np.testing.assert_allclose(d, [[1, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0]], atol=1e-12)
    d = RaySensor.pattern(3, 90.0, [0.0, 30.0])
    assert d.shape == (6, 3)
    az = np.degrees(np.arctan2(d[:, 1], d[:, 0]))
    np.testing.assert_allclose(az, [-45, 0, 45, -45, 0, 45], atol=1e-9)
    el = np.degrees(np.arcsin(d[:, 2]))
    np.testing.assert_allclose(el, [0, 0, 0, 30, 30, 30], atol=1e-9)
    np.testing.assert_allclose(np.linalg.norm(d, axis=1), 1.0)
    np.testing.assert_allclose(RaySensor.pattern(1, 120.0, [0.0]), [[1, 0, 0]])


def test_explicit_directions_normalised_and_compiled():
    node = example_config(directions=[[2, 0, 0], [0, 0, -3], [1, 1, 0]])
    env = compile_config(node)
    lidar = env.models['r2d2'].addons['lidar']
    np.testing.assert_allclose(lidar.directions, [[1, 0, 0], [0, 0, -1], [2 ** -0.5, 2 ** -0.5, 0]])
    op = [o for o in env.builder.ops if o['type'] == KERNEL_OPS['RAY_SENSOR']][0]
    assert op['iargs'][1:] == [3, 1] and op['n_obs'] == 6
    assert op['iargs'][0] == env.models['r2d2'].body.frame(env.models['r2d2'].get_frame_id('head_swivel'))
    np.testing.assert_allclose(np.reshape(op['fargs'][9:], (3, 3)), lidar.directions)
    np.testing.assert_allclose(op['fargs'][7:9], [0.05, 8.0])


def test_spaces_and_flattened_size():
    env = compile_config(example_config())
    sp = env.observation_space['r2d2']['lidar']
    assert sp['distance'].shape == (64, ) and sp['hit_object'].shape == (64, )
    assert np.all(sp['distance'].low == np.float32(0.05)) and np.all(sp['distance'].high == np.float32(8.0))
    assert env.scene.hdr['n_obs'] == 128
    node = example_config(include_hit_object=False, num_rays=64, vertical_angles=[0, -10])
    node['flatten_observations'] = True
    env = compile_config(node)
    assert env.observation_space.shape == (128, ) and env.scene.hdr['n_obs'] == 128


def test_scenes_without_the_sensor_compile_as_before():
    a = DIYGym(maze_with_lidar(False), num_envs=1, compile_only=True).scene
    b = DIYGym(os.path.join(ROOT, 'examples', 'r2d2_maze', 'r2d2_maze.yaml'), num_envs=1, compile_only=True).scene
    assert np.array_equal(a.ibuf, b.ibuf) and np.array_equal(a.fbuf, b.fbuf)


def test_op_code_and_generated_headers():
    """The ray op's code is defined beside its kernel and continues the generated numbering; the generated headers do not
    carry it (the step kernel and the oracle skip the op)."""
    with open(os.path.join(ROOT, 'diy_gym_b200', 'csrc', 'dg_ray.cuh')) as f:
        assert '#define OP_RAY_SENSOR %d\n' % KERNEL_OPS['RAY_SENSOR'] in f.read()
    for path in ('diy_gym_b200/csrc/scene_sections.h', 'oracle/scene_sections.h'):
        with open(os.path.join(ROOT, path)) as f:
            assert f.read() == emit_c_header()
    assert KERNEL_OPS['RAY_SENSOR'] == max(OP.values()) + 1


@pytest.mark.parametrize('edit', [dict(range=[-0.1, 5.0]), dict(range=[2.0, 2.0]), dict(range=[3.0, 1.0]), dict(num_rays=0),
                                  dict(horizontal_fov=0), dict(horizontal_fov=400), dict(directions=[[1, 0, 0], [0, 0, 0]]),
                                  dict(frame='no_such_joint'), dict(num_rays=1025), dict(num_rays=512, vertical_angles=[0, 1, 2])])
def test_invalid_configurations_raise(edit):
    with pytest.raises(ValueError):
        compile_config(example_config(**edit))


def test_environment_level_sensor_rejects_a_frame():
    node = example_config()
    node['world_lidar'] = dict(addon='ray_sensor', frame='head_swivel', num_rays=8)
    with pytest.raises(ValueError):
        compile_config(node)


def test_host_layer_on_emulated_world_nested_flattened_and_terminal_observation():
    from tests.emul.ray_emul import factory
    env = DIYGym(Configuration.from_dict('ray_sensor', example_config()), num_envs=2, world_factory=factory())
    obs = env.reset()
    d, h = obs['r2d2']['lidar']['distance'], obs['r2d2']['lidar']['hit_object']
    assert d.shape == (2, 64) and h.shape == (2, 64)
    assert float(d.min()) > 0.05 and float(d.max()) <= 8.0
    assert ((h >= -1) & (h < len(env.scene.bodies))).all() and (h >= 0).any()
    assert torch.equal(d[h < 0], torch.full_like(d[h < 0], 8.0))
    # flattened
    node = example_config()
    node['flatten_observations'] = True
    envf = DIYGym(Configuration.from_dict('ray_sensor', node), num_envs=2, world_factory=factory())
    flat = envf.reset()
    assert flat.shape == (2, 128)
    assert torch.equal(flat, torch.cat([d, h], dim=1))
    # auto_reset: the terminal observation carries the rays of the final step (a copy: the reset rewrites the rows)
    node = example_config()
    node['max_episode_steps'] = 2
    enva = DIYGym(Configuration.from_dict('ray_sensor', node), num_envs=2, world_factory=factory(), auto_reset=True)
    envb = DIYGym(Configuration.from_dict('ray_sensor', node), num_envs=2, world_factory=factory())
    act = {'r2d2': {'wheel_driver': torch.full((2, 4), 0.5)}}
    for _ in range(2):
        obs_a, _, _, info = enva.step(act)
        obs_b = envb.step(act)[0]
    assert bool(info['done'].all())
    term = info['terminal_observation']['r2d2']['lidar']
    assert torch.equal(term['distance'], obs_b['r2d2']['lidar']['distance'])
    assert torch.equal(term['hit_object'], obs_b['r2d2']['lidar']['hit_object'])
    assert torch.equal(obs_a['r2d2']['lidar']['distance'], enva.world.obs[:, :64])   # the rays of the fresh episode


# ---------------------------------------------------------------- known answers of the fp64 reference --------------
URDF = '''<robot name="k"><link name="base"><inertial><mass value="1"/><inertia ixx="1" ixy="0" ixz="0" iyy="1" iyz="0" izz="1"/></inertial>
<collision><origin xyz="0 0 0" rpy="0 0 0"/><geometry>%s</geometry></collision></link></robot>'''


def _kat_scene(tmp_path, targets, dirs, rng=(0.0, 10.0)):
    """A collision-free free body carrying the sensor (frame: its base) and static single-shape bodies."""
    sb = SceneBuilder()
    sensor = sb.add_body('sensor', resolve_model('sphere2red_nocol.urdf'))
    for i, (geom, xyz) in enumerate(targets):
        p = tmp_path / ('kat_%d_%s.urdf' % (i, abs(hash((geom, tuple(xyz), str(tmp_path))))))
        p.write_text(URDF % geom)
        sb.add_body('t%d' % i, resolve_model(str(p)), xyz=xyz, fixed_base=True)
    dirs = np.asarray(dirs, float)
    dirs = dirs / np.linalg.norm(dirs, axis=1, keepdims=True)
    sb.add_op('RAY_SENSOR', [sensor.frame(-1), len(dirs), 1], [0, 0, 0, 0, 0, 0, 1, rng[0], rng[1]] + dirs.reshape(-1).tolist(),
              n_obs=2 * len(dirs))
    return sb.finalize()


def _cast(scene, origin, quat=(0, 0, 0, 1)):
    """Distances and hit ids of the fp64 reference, with the fp32 device routines (g++ build) checked against them."""
    o = OracleWorld(scene)
    o.s('S_BPOS', 3)[:] = origin
    o.s('S_BQUAT', 4)[:] = quat
    o.refresh()
    obs = ray_reference.cast(scene, o.state)
    em = RayCaster(scene).rays(o.state)[0]
    R = len(obs) // 2
    np.testing.assert_allclose(em[:R], obs[:R], atol=2e-5, rtol=1e-5)
    np.testing.assert_array_equal(em[R:], obs[R:])
    return obs[:R], obs[R:]


def test_known_answers_primitives(tmp_path):
    targets = [('<box size="0.2 4 4"/>', (3, 0, 0)),                      # body 1: face at x = 2.9
               ('<sphere radius="0.5"/>', (0, 4, 0)),                     # body 2: surface at y = 3.5
               ('<cylinder radius="0.3" length="1.0"/>', (0, -3, 0)),      # body 3: side at y = -2.7, caps at z = +-0.5
               ('<capsule radius="0.2" length="0.8"/>', (-3, 0, 0))]      # body 4: end cap pole at z = 0.6 above its centre
    dirs = [[1, 0, 0], [0, 1, 0], [0, -1, 0], [-1, 0, 0], [0, 0, 1]]
    sc = _kat_scene(tmp_path, targets, dirs)
    d, h = _cast(sc, (0, 0, 0))
    np.testing.assert_allclose(d, [2.9, 3.5, 2.7, 2.8, 10.0], atol=1e-12)
    np.testing.assert_array_equal(h, [1, 2, 3, 4, -1])
    # cylinder cap from above and capsule end from above
    sc2 = _kat_scene(tmp_path, targets, [[0, 0, -1]])
    d, h = _cast(sc2, (0, -3, 3))
    np.testing.assert_allclose(d, [2.5], atol=1e-12)
    np.testing.assert_array_equal(h, [3])
    d, h = _cast(sc2, (-3, 0, 3))
    np.testing.assert_allclose(d, [3 - 0.4 - 0.2], atol=1e-12)
    np.testing.assert_array_equal(h, [4])
    # an oblique ray onto the sphere: |o + t u - c| = r
    u = np.array([0.1, 1.0, 0.05]) / np.linalg.norm([0.1, 1.0, 0.05])
    sc3 = _kat_scene(tmp_path, targets, [u])
    d, _ = _cast(sc3, (-0.5, 0, 0))
    oc = np.array([-0.5, -4, 0])
    b = oc @ u
    np.testing.assert_allclose(d, [-b - np.sqrt(b * b - (oc @ oc - 0.25))], atol=1e-12)


def test_min_hides_near_shapes_and_inside_origins_report_nothing(tmp_path):
    targets = [('<box size="0.2 4 4"/>', (3, 0, 0)), ('<box size="0.2 4 4"/>', (6, 0, 0)),
               ('<cylinder radius="0.3" length="1.0"/>', (0, -3, 0))]
    # min beyond the first wall: the second one (face at x = 5.9)
    d, h = _cast(_kat_scene(tmp_path, targets, [[1, 0, 0]], rng=(3.2, 10.0)), (0, 0, 0))
    np.testing.assert_allclose(d, [5.9], atol=1e-12)
    np.testing.assert_array_equal(h, [2])
    # the point at min inside the first wall: that wall is not reported
    d, h = _cast(_kat_scene(tmp_path, targets, [[1, 0, 0]], rng=(3.0, 10.0)), (0, 0, 0))
    np.testing.assert_allclose(d, [5.9], atol=1e-12)
    np.testing.assert_array_equal(h, [2])
    # inside the cylinder, looking up and sideways: nothing (the cap test alone would report the exit cap at 0.5)
    d, h = _cast(_kat_scene(tmp_path, targets, [[0, 0, 1], [0, 0, -1], [0, 1, 0]], rng=(0.0, 2.0)), (0, -3, 0.1))
    np.testing.assert_allclose(d, [2.0, 2.0, 2.0])
    np.testing.assert_array_equal(h, [-1, -1, -1])
    # a miss: max, id -1
    d, h = _cast(_kat_scene(tmp_path, targets, [[0, 0, 1]], rng=(0.1, 7.5)), (0, 0, 0))
    np.testing.assert_allclose(d, [7.5])
    np.testing.assert_array_equal(h, [-1])


def _plane_clip(planes, o, u):
    """numpy Cyrus-Beck: entry parameter of the ray o + t u into {x: n.x <= c} (None: no entry at t > 0)."""
    te, tx = -np.inf, np.inf
    for n, c in zip(planes[:, :3], planes[:, 3]):
        den, num = n @ u, c - n @ o
        if abs(den) < 1e-18:
            if num < 0:
                return None
            continue
        t = num / den
        if den < 0:
            te = max(te, t)
        else:
            tx = min(tx, t)
    return te if te <= tx and te > 0 else None


def test_ur5_hull_link_matches_numpy_plane_clip():
    sb = SceneBuilder()
    sensor = sb.add_body('sensor', resolve_model('sphere2red_nocol.urdf'))
    sb.add_body('arm', resolve_model('ur5/ur5_robot.urdf'), fixed_base=True)
    rng = np.random.default_rng(3)
    dirs = rng.normal(size=(48, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    sb.add_op('RAY_SENSOR', [sensor.frame(-1), 1, 1], [0, 0, 0, 0, 0, 0, 1, 0.0, 5.0, 1.0, 0.0, 0.0], n_obs=2)
    sc = sb.finalize()
    SI, SF, H = sc.sec['SHAPE_I'], sc.sec['SHAPE_F'], sc.sec['HULL_F']
    hulls = [s for s in range(len(SI)) if SI[s, 5] > 0]
    assert hulls
    o = OracleWorld(sc)
    o.refresh()
    agree = total = 0
    for s in hulls[1:4]:
        fs = o.frame_state(int(SI[s, 1]))
        Rf, pf = quat_to_mat(fs['com_quat']), fs['com_pos']
        R, p = Rf @ quat_to_mat(SF[s, 3:7]), pf + Rf @ SF[s, 0:3]
        planes = H[SI[s, 6]:SI[s, 6] + 4 * SI[s, 7]].reshape(-1, 4)
        verts = H[SI[s, 4]:SI[s, 4] + 3 * SI[s, 5]].reshape(-1, 3)
        c = verts.mean(axis=0)
        for u in dirs:
            # start 3 cm outside the hull along u (shape frame), look back at its centre
            t_out = min((pl[3] - pl[:3] @ c) / (pl[:3] @ u) for pl in planes if pl[:3] @ u > 1e-12)
            ol = c + (t_out + 0.03) * u
            ow, uw = p + R @ ol, -(R @ u)
            expect = _plane_clip(planes, ol, -u)
            assert expect is not None and abs(expect - 0.03) < 1e-9
            # sensor pose: the base of the free body at ow, its x axis along uw
            x = uw
            y = np.cross([0, 0, 1.0], x) if abs(x[2]) < 0.9 else np.cross([0, 1.0, 0], x)
            y /= np.linalg.norm(y)
            M = np.stack([x, y, np.cross(x, y)], axis=1)
            o.s('S_BPOS', 3)[:] = ow
            o.s('S_BQUAT', 4)[:] = mat_to_quat(M)
            o.refresh()
            d, hb = ray_reference.cast(sc, o.state)
            assert hb == 1 and d <= expect + 1e-9   # the arm, never behind this hull's surface
            agree += abs(d - expect) < 1e-9
            total += 1
    assert agree >= 0.8 * total, (agree, total)


def test_hit_ids_and_sensor_on_head_swivel_turns_with_q(tmp_path):
    sb = SceneBuilder()
    r2 = sb.add_body('r2d2', resolve_model('r2d2.urdf'), xyz=(0, 0, 0.5))
    for i, xyz in enumerate([(4, 0, 0), (0, 4, 0)]):
        p = tmp_path / ('wall_%d.urdf' % i)
        p.write_text(URDF % '<box size="0.2 0.2 4"/>')
        sb.add_body('w%d' % i, resolve_model(str(p)), xyz=xyz, fixed_base=True)
    head = r2.joint_index('head_swivel')
    sb.add_op('RAY_SENSOR', [r2.frame(head), 1, 1], [0.3, 0, 0.45, 0, 0, 0, 1, 0.05, 8.0, 1, 0, 0], n_obs=2)
    sc = sb.finalize()
    o = OracleWorld(sc)
    dof = r2.global_dof(head)
    out = {}
    for q in (0.0, np.pi / 2, np.pi):
        o.s('S_Q', sc.hdr['nd'])[dof] = q
        o.refresh()
        link = o.frame_state(r2.frame(head))
        R, pos = quat_to_mat(link['link_quat']), link['link_pos']
        org = pos + R @ [0.3, 0, 0.45]
        d, hb = ray_reference.cast(sc, o.state)
        out[q] = (d, hb, org)
        em = RayCaster(sc).rays(o.state)[0]
        assert abs(em[0] - d) < 2e-5 and em[1] == hb
    d, hb, org = out[0.0]
    assert hb == 1 and abs(d - (3.9 - org[0])) < 1e-9
    d, hb, org = out[np.pi / 2]
    assert hb == 2 and abs(d - (3.9 - org[1])) < 1e-9
    d, hb, _ = out[np.pi]
    assert hb == -1 and d == 8.0


# ---------------------------------------------------------------- emulation / kernel against the fp64 reference -----
def parity(scene, states, obs):
    """Every ray of every environment against the fp64 reference from the same state row.  A ray agrees when its distance is within
    1e-4 + 1e-5 d of the reference's and, where the op reports hit objects, its body index is the reference's.  Returns the fraction of
    agreeing rays, the number of id flips among distance-agreeing rays (a ray through the seam of two touching bodies hits both at
    the same distance: fp32 and fp64 may pick different ones) and the worst distance error."""
    good = total = flips = 0
    worst = (0.0, None)
    for e in range(len(states)):
        ref = ray_reference.cast(scene, states[e])
        for off, R, hit in ray_ops(scene):
            d, dr = obs[e, off:off + R], ref[off:off + R]
            err = np.abs(d - dr)
            ok = err <= 1e-4 + 1e-5 * dr
            if hit:
                same = obs[e, off + R:off + 2 * R] == ref[off + R:off + 2 * R]
                flips += int((ok & ~same).sum())
                ok &= same
            good += int(ok.sum())
            total += R
            k = int(np.argmax(err))
            if err[k] > worst[0]:
                worst = (float(err[k]), (e, off + k, float(d[k]), float(dr[k])))
    return good / total, flips, worst


def _emul_run(cfg, n, steps, seed=5):
    env = DIYGym(cfg, num_envs=1, compile_only=True)
    sc = env.scene
    e, rays = EmulWorld(sc, n, team=4, seed=seed), RayCaster(sc)
    e.reset()
    yield sc, e.state.copy(), rays.rays(e.state)
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        e.step(rng.uniform(-0.5, 0.5, size=(n, sc.hdr['n_act'])).astype(np.float32))
    yield sc, e.state.copy(), rays.rays(e.state)


@pytest.mark.parametrize('which', ['example', 'maze_lidar'])
def test_emulation_matches_reference_after_reset_and_random_steps(which):
    cfg = Configuration.from_dict('ray_sensor', example_config()) if which == 'example' else maze_with_lidar(**MAZE_LIDAR)
    for sc, st, ob in _emul_run(cfg, 3, 10):
        frac, flips, worst = parity(sc, st, ob)
        print('%s: %.5f of the rays agree (%d id flips), worst distance error %s' % (which, frac, flips, worst))
        assert frac >= 0.999, worst


# ---------------------------------------------------------------- GPU -----------------------------------------------
def _gpu_world(cfg, n, **kw):
    from diy_gym_b200.backend import World
    sc = DIYGym(cfg, num_envs=1, compile_only=True).scene
    return sc, World(sc, n, **kw)


def _rays(sc, obs):
    cols = np.concatenate([np.arange(off, off + (2 * R if hit else R)) for off, R, hit in ray_ops(sc)])
    return obs[:, cols]


@pytest.mark.gpu
@pytest.mark.parametrize('which,n,sample', [('maze_lidar', 4096, 64), ('example', 64, 64)])
def test_gpu_kernel_matches_reference(which, n, sample):
    cfg = Configuration.from_dict('ray_sensor', example_config()) if which == 'example' else maze_with_lidar(**MAZE_LIDAR)
    sc, w = _gpu_world(cfg, n, seed=11)
    w.reset()
    pick = np.random.default_rng(0).choice(n, size=min(sample, n), replace=False)
    for leg in ('reset', 'steps'):
        if leg == 'steps':
            g = torch.Generator(device=w.device).manual_seed(1)
            for _ in range(10):
                w.action.copy_(torch.rand(w.action.shape, generator=g, device=w.device) - 0.5)
                w.step()
        torch.cuda.synchronize()
        st, ob = w.state.cpu().numpy()[pick], w.obs.cpu().numpy()[pick]
        frac, flips, worst = parity(sc, st, ob)
        print('%s %s: %.5f of the rays agree (%d id flips), worst distance error %s' % (which, leg, frac, flips, worst))
        assert frac >= 0.999, worst
    w.close()


@pytest.mark.gpu
@pytest.mark.parametrize('split', ['0', '1'])
def test_gpu_observe_after_step_rewrites_rays_bit_identically(monkeypatch, split):
    monkeypatch.setenv('DG_SPLIT', split)
    sc, w = _gpu_world(maze_with_lidar(**MAZE_LIDAR), 1000, seed=3)
    w.reset()
    w.action.uniform_(-0.5, 0.5)
    for _ in range(5):
        w.step()
    after_step = w.obs.clone()
    w.obs.fill_(-7.0)
    w.observe()
    torch.cuda.synchronize()
    assert torch.equal(after_step, w.obs)
    w.close()


@pytest.mark.gpu
def test_gpu_graph_replay_matches_plain_launches(monkeypatch):
    monkeypatch.setenv('DG_SPLIT', '1')
    out = []
    for graph in ('0', '1'):
        monkeypatch.setenv('DG_GRAPH', graph)
        sc, w = _gpu_world(maze_with_lidar(**MAZE_LIDAR), 512, seed=9)
        w.reset()
        g = torch.Generator(device=w.device).manual_seed(2)
        obs = []
        for _ in range(20):
            w.action.copy_(torch.rand(w.action.shape, generator=g, device=w.device) - 0.5)
            w.step()
            obs.append(w.obs.clone())
        torch.cuda.synchronize()
        out.append(torch.stack(obs))
        w.close()
    assert torch.equal(out[0], out[1])


@pytest.mark.gpu
def test_gpu_step_host_equals_step_plus_copies():
    cfg = Configuration.from_dict('ray_sensor', example_config())
    (sc, a), (_, b) = _gpu_world(cfg, 96, seed=4), _gpu_world(cfg, 96, seed=4)
    a.reset()
    b.reset()
    rng = np.random.default_rng(0)
    for _ in range(5):
        act = rng.uniform(-0.5, 0.5, size=(96, sc.hdr['n_act'])).astype(np.float32)
        a.action.copy_(torch.from_numpy(act))
        a.step()
        o = np.zeros((96, sc.hdr['n_obs']), np.float32)
        r = np.zeros((96, max(sc.hdr['n_rew'], 0)), np.float32)
        t = np.zeros((96, max(sc.hdr['n_term'], 0)), np.uint8)
        b.step_host(act, o, r, t)
        torch.cuda.synchronize()
        assert np.array_equal(a.obs.cpu().numpy(), o)
    a.close()
    b.close()


@pytest.mark.gpu
def test_gpu_masked_reset_only_changes_masked_rays():
    sc, w = _gpu_world(maze_with_lidar(**MAZE_LIDAR), 300, seed=8)
    w.reset()
    w.action.uniform_(-0.5, 0.5)
    for _ in range(10):
        w.step()
    torch.cuda.synchronize()
    before = w.obs.clone()
    mask = torch.zeros(300, dtype=torch.uint8)
    mask[::3] = 1
    w.reset(mask)
    torch.cuda.synchronize()
    m = mask.bool().to(w.device)
    assert torch.equal(before[~m], w.obs[~m])
    assert not torch.equal(before[m], w.obs[m])
    w.close()


@pytest.mark.gpu
def test_gpu_hundred_rays_and_two_sensors_on_a_partial_block():
    node = example_config(num_rays=100, vertical_angles=[0], include_hit_object=False)
    node['world_lidar'] = dict(addon='ray_sensor', xyz=[0.5, -0.5, 0.8], num_rays=40, horizontal_fov=270, vertical_angles=[-5, 5],
                               range=[0.1, 6.0], include_hit_object=True)
    n = 37
    sc, w = _gpu_world(Configuration.from_dict('ray_sensor', node), n, seed=6)
    assert sorted((R, hit) for _, R, hit in ray_ops(sc)) == [(80, True), (100, False)]
    w.reset()
    w.action.uniform_(-0.5, 0.5)
    for _ in range(3):
        w.step()
    torch.cuda.synchronize()
    frac, flips, worst = parity(sc, w.state.cpu().numpy(), w.obs.cpu().numpy())
    assert frac >= 0.999, worst
    w.close()
