"""The camera kernel (dg_render_kernel<NCW, NH, U8> in csrc/dg_kernels.cu) against the fp64 reference of tests/camera_reference.py,
in every instantiation and store path it has.

Synthetic scenes (temporary URDFs): a fixed-base body whose visuals are baked into the scene tables, a floating body with several
links (moving visuals), a camera on one of its links and one fixed in the world.  Every environment gets its own random pose of
the floating body and its links, written straight into the state row, and its own colours in the parameter row.  The number of
visual shapes sets the candidate words (NCW 1: up to 32, 2: up to 64, 4: more, with a per-shape tail above 128); the image size
sets the patch height (NH) and which stores run (whole 16-byte pieces of staged patches, or pixel by pixel); the batch size sets
how many blocks render one image (`groups`).  `launch_config` restates that choice and test_matrix_reaches_every_instantiation
checks that CASES reach all of it.

On the CPU the reference is checked against the oracle's ray caster (dgo_render_seg).  On the GPU every case renders float
colour with the mask and byte colour with the mask, into buffers filled with NaN / 0xAB first, and off the reference's ambiguity
mask requires the same mask; off it and off the grazing hits (camera_reference.render) depth and colour within the bars below,
bytes = round(255 clamp(colour)) except where the colour error can reach a rounding tie; everywhere, depth and mask of the byte render bit-identical to
the float render."""
import ctypes
import os
import tempfile

import numpy as np
import pytest

from diy_gym_b200.compiler.mathutil import mat_to_quat, quat_from_euler, quat_to_mat
from diy_gym_b200.compiler.scene import SceneBuilder
from diy_gym_b200.compiler.urdf import compile_urdf
from tests import camera_reference as cref

EX = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'examples')

# Bars off the ambiguity and grazing masks: depth within DEPTH_RTOL relative plus DEPTH_ULPS times the bound on one fp32 rounding
# of the terms of ray_shape's discriminant B^2 - A C, colour within RGB_ATOL plus RGB_ULPS times the same bound carried to the
# colour (camera_reference.entry).  The bound matters for small spheres, capsules and cylinders seen from afar, where the
# discriminant cancels by (distance / radius)^2; boxes and caps get the fixed bars only.  The colour term leaves out the rounding
# of the normal's own arithmetic, so it takes the larger multiple.  Worst seen on a B200 (1000 W): 0.57 of the depth bar and 0.77
# of the colour bar; in absolute terms depth 6.5e-5 relative and colour 1.0e-3, both where the bound term is large.
DEPTH_RTOL = 2e-5
RGB_ATOL = 1e-4
DEPTH_ULPS = 4
RGB_ULPS = 32
B200_SMS = 148
TYPES = ('box', 'sphere', 'cylinder', 'capsule')
STATE_SEEDS = 8      # distinct states in the large batch

# (visual shapes, (camera 0 on the floating body, camera 1 in the world) as (width, height), environments); 'big' = 8 SMs + 3
CASES = [
    (31, ((1, 1), (200, 200)), 3),
    (32, ((7, 3), (96, 64)), 1),
    (33, ((8, 4), (160, 90)), 37),
    (64, ((88, 64), (100, 60)), 3),
    (65, ((88, 64), (100, 60)), 'big'),
    (128, ((90, 90), (160, 90)), 3),
    (129, ((8, 4), (96, 64)), 37),
    (240, ((88, 64), (200, 200)), 3),
    (300, ((1, 1), (160, 90)), 3),
]


def n_envs(n, sms):
    return 8 * sms + 3 if n == 'big' else n


# ---------------------------------------------------------------- launch configuration ----------------------------------------
def launch_config(width, height, nv, n, sms, u8):
    """What render_any (csrc/dg_kernels.cu) launches: NCW (render_kernel), NH, U8, vec_ok and groups, and the store paths the
    patches take (dg_render_kernel: a patch is staged when vec_ok and it is 8 pixels wide; a staged patch is cut short at the
    bottom when the image ends inside it; the rest is stored pixel by pixel, 'scalar_right' when the image itself is staged)."""
    nh = 2 if ((width + 7) // 8) * ((height + 7) // 8) >= 96 else 1
    ncw = (nv + 31) // 32
    ncw = 1 if ncw <= 1 else (2 if ncw == 2 else 4)
    tiles_x, tiles_y = (width + 7) // 8, (height + 4 * nh - 1) // (4 * nh)
    groups = max(1, min((tiles_x * tiles_y + 7) // 8, (8 * sms + n - 1) // n))
    vec_ok = width % (8 if u8 else 4) == 0
    mt_h, paths = 4 * nh, set()
    for py0 in range(0, height, mt_h):
        for px0 in range(0, width, 8):
            if vec_ok and min(8, width - px0) == 8:
                paths.add('staged' if min(mt_h, height - py0) == mt_h else 'staged_bottom')
            else:
                paths.add('scalar_right' if vec_ok else 'scalar')
    return dict(ncw=ncw, nh=nh, u8=u8, vec_ok=vec_ok, groups=groups, paths=paths)


def test_matrix_reaches_every_instantiation():
    kernels, paths, groups = set(), set(), set()
    for nv, cams, n in CASES:
        for (w, h) in cams:
            for u8 in (False, True):
                c = launch_config(w, h, nv, n_envs(n, B200_SMS), B200_SMS, u8)
                kernels.add((c['ncw'], c['nh'], c['u8']))
                paths |= {(c['nh'], c['u8'], p) for p in c['paths']}
                groups.add(c['groups'] > 1)
    assert kernels == {(a, b, c) for a in (1, 2, 4) for b in (1, 2) for c in (False, True)}
    for nh in (1, 2):
        for u8 in (False, True):
            assert (nh, u8, 'staged') in paths and (nh, u8, 'scalar') in paths, (nh, u8)
    assert (2, False, 'staged_bottom') in paths and (2, True, 'staged_bottom') in paths
    assert (2, False, 'scalar_right') in paths                 # 100 x 60: staged float with a partial right patch ...
    assert launch_config(100, 60, 64, 3, B200_SMS, True)['paths'] == {'scalar'}   # ... and scalar bytes
    assert groups == {False, True}
    # the shape counts around each boundary, and the tail loop above 128
    assert {31, 32, 33, 64, 65, 128, 129, 240, 300} <= {nv for nv, _, _ in CASES}


def test_launch_config_of_the_example_cameras():
    """The two example cameras: 50 x 50 (8 x 4 patches, every pixel scalar) and 200 x 200 (8 x 8 patches, all staged)."""
    a = launch_config(50, 50, 20, 2, B200_SMS, False)
    b = launch_config(200, 200, 20, 2, B200_SMS, True)
    assert (a['nh'], a['ncw'], a['paths']) == (1, 1, {'scalar'}) and a['groups'] > 1
    assert (b['nh'], b['ncw'], b['paths']) == (2, 1, {'staged'}) and b['groups'] > 1


# ---------------------------------------------------------------- synthetic scenes ---------------------------------------------
def _geom(kind, dims):
    if kind == 'box':
        return '<box size="%.17g %.17g %.17g"/>' % tuple(2 * d for d in dims[:3])
    if kind == 'sphere':
        return '<sphere radius="%.17g"/>' % dims[0]
    return '<%s radius="%.17g" length="%.17g"/>' % (kind, dims[0], 2 * dims[1])


def _visual(kind, dims, xyz, rpy, rgba=(0.8, 0.8, 0.8, 1)):
    return ('<visual><origin xyz="%.17g %.17g %.17g" rpy="%.17g %.17g %.17g"/><geometry>%s</geometry><material name=""><color rgba="%.17g %.17g %.17g %.17g"/>'
            '</material></visual>' % (tuple(xyz) + tuple(rpy) + (_geom(kind, dims), ) + tuple(rgba)))


def _link(name, visuals, inertial_xyz=(0, 0, 0), inertial_rpy=(0, 0, 0)):
    return ('<link name="%s"><inertial><origin xyz="%.17g %.17g %.17g" rpy="%.17g %.17g %.17g"/><mass value="1"/><inertia ixx="0.01" iyy="0.01" '
            'izz="0.01" ixy="0" ixz="0" iyz="0"/></inertial>%s</link>' % ((name, ) + tuple(inertial_xyz) + tuple(inertial_rpy) + (''.join(visuals), )))


def _urdf(path, name, links, joints):
    with open(path, 'w') as f:
        f.write('<?xml version="1.0"?><robot name="%s">%s%s</robot>' % (name, ''.join(links), ''.join(
            '<joint name="j%d" type="fixed"><parent link="%s"/><child link="%s"/><origin xyz="%.17g %.17g %.17g"/></joint>' % ((k, p, c) + tuple(o))
            for k, (p, c, o) in enumerate(joints))))
    return compile_urdf(path)


def _random_visuals(rng, n, radius):
    out = []
    for k in range(n):
        kind = TYPES[k % 4]
        dims = list(rng.uniform(0.03, 0.16, 3))
        xyz = rng.normal(size=3)
        xyz = xyz / np.linalg.norm(xyz) * radius * rng.uniform(0.1, 1.0) ** (1 / 3)
        out.append(_visual(kind, dims, xyz, rng.uniform(-np.pi, np.pi, 3), tuple(rng.uniform(0, 1, 3)) + (1, )))
    return out


def look_at(eye, target, roll):
    """Camera rotation (columns: right, up, backward; the camera looks along -z) from `eye` towards `target`, rolled by `roll`."""
    z = np.asarray(eye, float) - target
    z /= np.linalg.norm(z)
    x = np.cross([0.0, 0.0, 1.0], z)
    x = x / np.linalg.norm(x) if np.linalg.norm(x) > 1e-9 else np.array([1.0, 0, 0])
    y = np.cross(z, x)
    R = np.stack([x, y, z], axis=1)
    c, s = np.cos(roll), np.sin(roll)
    return R @ np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])


CAM_XYZ, CAM_RPY = (0.05, -0.02, 0.1), (0.3, -0.2, 0.4)     # camera 0 in the URDF frame of its link
CAM_LINK_INERTIAL = ((0.02, 0.03, -0.04), (0.1, 0.2, -0.3))


def synthetic_scene(nv, cams, tmp, seed=0, fov=(60.0, 75.0), near=0.05, far=8.0):
    """nv visual shapes: about half on a fixed-base body (baked), the rest on three links of a floating body, plus camera 0 on
    the floating body's fourth link and camera 1 fixed in the world, looking at the origin with a roll."""
    rng = np.random.default_rng(1000 + nv + seed)
    n_static = nv // 2
    n_move = nv - n_static
    per = [n_move // 3 + (1 if k < n_move % 3 else 0) for k in range(3)]
    static = _urdf(os.path.join(tmp, 'static_%d.urdf' % nv), 'static', [_link('base', _random_visuals(rng, n_static, 1.0))], [])
    links = [_link('l%d' % k, _random_visuals(rng, per[k], 0.35)) for k in range(3)]
    links.append(_link('cam', [], *CAM_LINK_INERTIAL))
    rig = _urdf(os.path.join(tmp, 'rig_%d.urdf' % nv), 'rig', links, [('l0', 'l1', (0.1, 0, 0)), ('l1', 'l2', (0, 0.1, 0)), ('l0', 'cam', (0, 0, 0.2))])
    sb = SceneBuilder()
    sb.add_body('static', static, fixed_base=True)
    b = sb.add_body('rig', rig, xyz=(0, 0, 0.3))
    sb.add_camera(b.frame(2), CAM_XYZ, quat_from_euler(CAM_RPY), cams[0][0], cams[0][1], fov[0], near, far)
    eye = np.array([2.2, -1.6, 1.1])
    sb.add_camera(-1, eye, mat_to_quat(look_at(eye, np.zeros(3), 0.35)), cams[1][0], cams[1][1], fov[1], near, far)
    return sb.finalize()


def _set_com_pose(sc, st, frame, R, p):
    h, nb = sc.hdr, sc.hdr['nb']
    if frame < nb:
        st[h['S_BPOS'] + 3 * frame:h['S_BPOS'] + 3 * frame + 3], st[h['S_BQUAT'] + 4 * frame:h['S_BQUAT'] + 4 * frame + 4] = p, mat_to_quat(R)
    else:
        gl = frame - nb
        st[h['S_LPOS'] + 3 * gl:h['S_LPOS'] + 3 * gl + 3], st[h['S_LQUAT'] + 4 * gl:h['S_LQUAT'] + 4 * gl + 4] = p, mat_to_quat(R)


def _random_rot(rng):
    q = rng.normal(size=4)
    return quat_to_mat(q / np.linalg.norm(q))


def random_rows(sc, rng):
    """A state row with random poses of every moving frame (camera 0's link placed so that the camera looks at the scene from
    2-3 m with a roll) and a parameter row with random colours, both float32 as the device keeps them."""
    st = np.array(sc.sec['STATE_DEFAULT'], np.float64)
    prm = np.array(sc.sec['PARAM_DEFAULT'], np.float64)
    for f in range(sc.hdr['nb'] + sc.hdr['nl']):
        if f < sc.hdr['nb'] and sc.sec['BODY_I'][f][7]:
            continue                                                 # baked: the kernel reads the compiled pose
        p = rng.normal(size=3)
        _set_com_pose(sc, st, f, _random_rot(rng), 0.3 * p / max(np.linalg.norm(p), 1e-9) * rng.uniform(0, 1))
    ci, cf = sc.sec['CAM_I'][0], sc.sec['CAM_F'][0]
    if ci[0] >= sc.hdr['nb']:
        d = rng.normal(size=3)
        eye = d / np.linalg.norm(d) * rng.uniform(2.0, 3.0)
        Rc = look_at(eye, rng.uniform(-0.2, 0.2, 3), rng.uniform(-np.pi, np.pi))
        Rl = Rc @ quat_to_mat(cf[3:7]).T                             # link frame = camera x offset^-1
        pl = eye - Rl @ cf[0:3]
        lf = sc.sec['LINK_F'][ci[0] - sc.hdr['nb']]
        Rcom = Rl @ quat_to_mat(lf[16:20])                           # COM frame = link frame x inertial frame
        _set_com_pose(sc, st, int(ci[0]), Rcom, pl + Rcom @ lf[7:10])
    nv = sc.hdr['nv']
    prm[sc.hdr['P_COLOR']:sc.hdr['P_COLOR'] + 3 * nv] = rng.uniform(0, 1, 3 * nv)
    return st.astype(np.float32), prm.astype(np.float32)


def edge_scene(tmp, cams=((64, 48), (160, 90))):
    """Geometry edges, one world camera each (cameras 0-4 at x = 0, 10, 20, 30, 40, all rolled), sharing one baked body:
      0: near = 0.5 with a box and a capsule crossing the near plane, shapes behind the eye, a sphere past far = 3 and a box across
         it, and two coincident spheres and boxes of two floating bodies (the lower index must win);
      1, 2, 3: the eye inside a sphere, a box, a cylinder (whose far cap it sees), with shapes around;
      4: near = 1e-3 with a box 2 mm in front of the eye."""
    vis = []
    # camera 0 looks along -z from (0, 0, 0): depth = -z
    vis += [_visual('box', (0.2, 0.15, 0.1), (0.1, 0.05, -0.5), (0.3, 0.2, 0.1)), _visual('capsule', (0.06, 0.2), (-0.15, -0.1, -0.5), (1.2, 0.3, 0)),
            _visual('sphere', (0.3, ), (0, 0, 1.0), (0, 0, 0)), _visual('box', (5, 5, 0.1), (0, 0, 2.0), (0, 0, 0)),
            _visual('sphere', (0.4, ), (0.3, 0.2, -4.0), (0, 0, 0)), _visual('box', (0.3, 0.2, 0.3), (-0.4, 0.2, -3.0), (0.4, 0.5, 0.6)),
            _visual('cylinder', (0.3, 0.5), (0, 0, -2.2), (1.5, 0, 0.3))]
    # 1: inside a sphere, 2: a box, 3: a cylinder (axis along the view direction), each with two shapes within it and one beyond
    for k, kind, dims in ((1, 'sphere', (0.8, )), (2, 'box', (0.7, 0.6, 0.9)), (3, 'cylinder', (0.7, 0.6))):
        x = 10.0 * k
        vis += [_visual(kind, dims, (x, 0.05, -0.02), (0, 0, 0)), _visual('sphere', (0.1, ), (x + 0.15, 0, -0.4), (0, 0, 0)),
                _visual('box', (0.08, 0.1, 0.05), (x - 0.2, 0.1, -0.3), (0.5, 0.1, 0.2)), _visual('capsule', (0.2, 0.3), (x, 0, -2.0), (0.2, 1.3, 0))]
    vis += [_visual('box', (0.5, 0.5, 0.05), (40.0, 0, -0.052), (0, 0, 0)), _visual('sphere', (0.3, ), (40.2, 0.1, -1.0), (0, 0, 0))]
    static = _urdf(os.path.join(tmp, 'edge_static.urdf'), 'static', [_link('base', vis)], [])
    twin = _urdf(os.path.join(tmp, 'twin.urdf'), 'twin', [_link('base', [_visual('sphere', (0.12, ), (0, 0, 0), (0, 0, 0)),
                                                                         _visual('box', (0.1, 0.08, 0.06), (0.1, 0, 0.05), (0.3, 0, 0))])], [])
    sb = SceneBuilder()
    sb.add_body('static', static, fixed_base=True)
    sb.add_body('twin_a', twin, xyz=(0.3, -0.25, -1.2))
    sb.add_body('twin_b', twin, xyz=(0.3, -0.25, -1.2))
    for k, (near, far) in enumerate(((0.5, 3.0), (0.05, 8.0), (0.05, 8.0), (0.05, 8.0), (1e-3, 8.0))):
        w, h = cams[k % 2]
        roll = 0.4 + 0.3 * k
        sb.add_camera(-1, (10.0 * k, 0, 0), quat_from_euler((0, 0, roll)), w, h, 70.0, near, far)
    return sb.finalize()


def edge_rows(sc, rng):
    """Both twins at the same random pose in front of camera 0, random colours."""
    st = np.array(sc.sec['STATE_DEFAULT'], np.float64)
    prm = np.array(sc.sec['PARAM_DEFAULT'], np.float64)
    R, p = _random_rot(rng), np.array([0.25, -0.2, -1.2]) + rng.uniform(-0.05, 0.05, 3)
    for f in (1, 2):
        _set_com_pose(sc, st, f, R, p)
    nv = sc.hdr['nv']
    prm[sc.hdr['P_COLOR']:sc.hdr['P_COLOR'] + 3 * nv] = rng.uniform(0, 1, 3 * nv)
    return st.astype(np.float32), prm.astype(np.float32)


# ---------------------------------------------------------------- the reference against the oracle (CPU) -------------------------
def _oracle_agrees(sc, st, prm, cam):
    from oracle.oracle import OracleWorld
    o = OracleWorld(sc)
    o.state[:], o.param[:] = st, prm
    rgb_o, depth_o, seg_o = o.render(cam, seg=True)
    ref = cref.render(sc, st, prm, cam)
    ok = ~ref['ambiguous']
    assert np.array_equal(ref['seg'][ok], seg_o[ok])
    assert (ref['allowed'] == seg_o[..., None]).any(axis=-1).all()
    same = ref['seg'] == seg_o
    assert np.abs(ref['depth'] - depth_o)[same].max() <= 1e-9
    assert np.abs(ref['rgb'] - rgb_o)[same].max() <= 1e-9
    return ref


@pytest.mark.parametrize('name', ['basic_env', 'from_the_readme'])
def test_reference_matches_oracle_on_examples(name):
    from diy_gym_b200 import DIYGym
    from tests.emul.world import factory
    env = DIYGym(os.path.join(EX, name, name + '.yaml'), num_envs=1, device=0, world_factory=factory(4))
    env.reset()
    for _ in range(5):
        env.world.step()
    st, prm = env.world.state[0].numpy().astype(np.float64), env.world.param[0].numpy().astype(np.float64)
    for cam in range(env.scene.hdr['ncam']):
        ref = _oracle_agrees(env.scene, st, prm, cam)
        assert (ref['seg'] >= 0).any() and ref['ambiguous'].mean() < 0.01
    env.close()


@pytest.mark.parametrize('nv', [31, 65, 129, 300])
def test_reference_matches_oracle_on_synthetic_scenes(nv):
    with tempfile.TemporaryDirectory() as tmp:
        sc = synthetic_scene(nv, ((40, 30), (48, 36)), tmp)
    rng = np.random.default_rng(nv)
    for _ in range(2):
        st, prm = random_rows(sc, rng)
        for cam in (0, 1):
            ref = _oracle_agrees(sc, st.astype(np.float64), prm.astype(np.float64), cam)
            assert len(np.unique(ref['seg'])) >= 2                 # something of the scene is in view


def test_reference_matches_oracle_on_geometry_edges():
    with tempfile.TemporaryDirectory() as tmp:
        sc = edge_scene(tmp, cams=((48, 36), (40, 30)))
    st, prm = edge_rows(sc, np.random.default_rng(5))
    refs = [_oracle_agrees(sc, st.astype(np.float64), prm.astype(np.float64), cam) for cam in range(sc.hdr['ncam'])]
    VI = sc.sec['VIS_I']
    seen = [set(np.unique(r['vis'])) for r in refs]
    # camera 0: the box crossing near is entered before near everywhere and so never seen, the capsule crossing it is seen where
    # its surface lies beyond near; the shapes behind the eye and past far are not seen, the box across far is; of the
    # coincident twins only the first body is seen
    assert 0 not in seen[0] and {1, 5, 6} <= seen[0] and not ({2, 3, 4} & seen[0])
    twins = [s for s in range(len(VI)) if VI[s, 3] in (1, 2)]
    assert {VI[s, 3] for s in seen[0] if s in twins} == {1}
    # cameras 1-3: the enclosing shape is invisible from inside, except the cylinder's far cap
    assert 7 not in seen[1] and 11 not in seen[2] and 15 in seen[3]
    assert {8, 9, 10} <= seen[1] and {12, 13, 14} <= seen[2] and {16, 17} <= seen[3]
    assert seen[4] == {19}                                           # 2 mm in front of the eye, beyond near = 1 mm


# ---------------------------------------------------------------- the kernel against the reference (GPU) -------------------------
def _fill_buffers(w, cam, u8):
    import torch
    wd, hg = w.cams[cam]
    N, dev = w.n_envs, w.device
    key = ('u8', cam) if u8 else cam
    w._img[key] = (torch.full((N, hg, wd, 3), 0xAB, dtype=torch.uint8, device=dev) if u8 else torch.full((N, hg, wd, 3), float('nan'), device=dev),
                   torch.full((N, hg, wd), float('nan'), device=dev))
    w._img[('seg', cam)] = torch.full((N, hg, wd), float('nan'), device=dev)


def render_both(w, cam):
    """(rgb, depth, seg) of the float render and (rgb bytes, depth, seg) of the byte render, as numpy, from NaN / 0xAB filled buffers."""
    import torch
    out = []
    for u8 in (False, True):
        _fill_buffers(w, cam, u8)
        res = w.render(cam, seg=True, u8=u8)
        torch.cuda.synchronize()
        out.append(tuple(t.cpu().numpy() for t in res))
    return out


def compare_env(sc, st, prm, cam, f, b, label, stats):
    ref = cref.render(sc, st.astype(np.float64), prm.astype(np.float64), cam)
    rgb, depth, seg = f
    rgb8, depth8, seg8 = b
    assert np.isfinite(rgb).all() and np.isfinite(depth).all() and np.isfinite(seg).all(), (label, 'unwritten pixels')
    assert np.array_equal(depth8.view(np.uint32), depth.view(np.uint32)) and np.array_equal(seg8, seg), label
    amb = ref['ambiguous']
    ok = ~amb
    bad = ok & (seg != ref['seg'])
    assert not bad.any(), (label, 'mask differs off the ambiguity mask at', np.argwhere(bad)[:5], seg[bad][:5], ref['seg'][bad][:5])
    assert (ref['allowed'] == seg[..., None]).any(axis=-1).all(), (label, 'ambiguous pixel with a mask value of no nearby ray')
    ill = ref['ill_conditioned']
    assert (amb | ill).sum() <= max(2, 0.01 * amb.size), (label, amb.mean(), ill.mean())
    derr = np.abs(depth.astype(np.float64) - ref['depth']) / np.abs(ref['depth'])
    cerr = np.abs(rgb.astype(np.float64) - ref['rgb']).max(axis=-1)
    ok = ok & ~ill                                                    # grazing hits: the same mask, depth and colour unbarred
    dbar = DEPTH_RTOL + DEPTH_ULPS * ref['depth_err'] / np.abs(ref['depth'])
    cbar = RGB_ATOL + RGB_ULPS * ref['rgb_err']
    dmax, cmax = float(derr[ok].max(initial=0)), float(cerr[ok].max(initial=0))
    dq, cq = float((derr / dbar)[ok].max(initial=0)), float((cerr / cbar)[ok].max(initial=0))
    # bytes: round(255 clamp(c)) of the reference, one off only where the kernel's colour error can reach a rounding tie; and
    # round(255 clamp(c)) of the float render (the same arithmetic in another instantiation), one off at most at its ties
    x = 255.0 * np.clip(ref['rgb'], 0, 1)
    tie = np.abs(x - np.floor(x) - 0.5) <= 255.0 * cerr[..., None]
    d8 = np.abs(rgb8.astype(np.float64) - np.rint(x))
    assert (d8[ok] <= np.where(tie, 1.0, 0.0)[ok]).all(), (label, 'bytes differ from round(255 c)')
    mine = np.rint(np.clip(rgb, 0, 1) * np.float32(255.0)).astype(np.float64)
    assert np.abs(rgb8 - mine).max(initial=0) <= 1 and (rgb8 != mine).mean() < 1e-3, (label, 'bytes differ from the float render')
    s = stats.setdefault(label, dict(depth_rel=0.0, rgb_abs=0.0, ambiguous=0.0, ill=0.0, ill_depth_rel=0.0, ill_rgb_abs=0.0, dq=0.0, cq=0.0))
    s['dq'], s['cq'] = max(s['dq'], dq), max(s['cq'], cq)
    s['depth_rel'], s['rgb_abs'], s['ambiguous'] = max(s['depth_rel'], dmax), max(s['rgb_abs'], cmax), max(s['ambiguous'], float(amb.mean()))
    s['ill'] = max(s['ill'], float(ill.mean()))
    s['ill_depth_rel'] = max(s['ill_depth_rel'], float(derr[ill].max(initial=0)))
    s['ill_rgb_abs'] = max(s['ill_rgb_abs'], float(cerr[ill].max(initial=0)))
    assert dq <= 1 and cq <= 1, (label, 'depth / colour error over the bar', dmax, dq, cmax, cq)


def _report(stats):
    for k, s in stats.items():
        print('camera-kernel %-40s worst depth rel %.2e (%.2f of its bar)  worst rgb abs %.2e (%.2f)  ambiguous %.4f  grazing %.4f '
              '(worst depth rel %.2e, rgb abs %.2e)' % (k, s['depth_rel'], s['dq'], s['rgb_abs'], s['cq'], s['ambiguous'], s['ill'],
                                                       s['ill_depth_rel'], s['ill_rgb_abs']))


@pytest.mark.gpu
@pytest.mark.parametrize('nv,cams,n', CASES, ids=['nv%d' % c[0] for c in CASES])
def test_camera_kernel_matches_reference(nv, cams, n):
    import torch
    from diy_gym_b200.backend import World
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = n_envs(n, sms)
    with tempfile.TemporaryDirectory() as tmp:
        sc = synthetic_scene(nv, cams, tmp)
    rng = np.random.default_rng(nv)
    K = min(N, STATE_SEEDS)
    rows = [random_rows(sc, rng) for _ in range(K)]
    which = np.arange(N) % K
    w = World(sc, N)
    w.state.copy_(torch.from_numpy(np.stack([rows[k][0] for k in which])))
    w.param.copy_(torch.from_numpy(np.stack([rows[k][1] for k in which])))
    stats = {}
    sample = list(range(K)) if n == 'big' else sorted({0, N - 1})
    for cam in (0, 1):
        f, b = render_both(w, cam)
        cfg = launch_config(cams[cam][0], cams[cam][1], nv, N, sms, False)
        label = 'nv%d cam%d %dx%d n=%d groups=%d' % (nv, cam, cams[cam][0], cams[cam][1], N, cfg['groups'])
        for e in sample:
            compare_env(sc, rows[which[e]][0], rows[which[e]][1], cam, tuple(a[e] for a in f), tuple(a[e] for a in b), label, stats)
        if N > K:      # the same state gives the same image, whatever block or group rendered it
            for a in f + b:
                assert np.array_equal(a.view(np.uint8), a[which].view(np.uint8)) if a.dtype == np.uint8 else np.array_equal(a.view(np.uint32), a[which].view(np.uint32))
    w.close()
    _report(stats)


@pytest.mark.gpu
def test_camera_kernel_geometry_edges():
    import torch
    from diy_gym_b200.backend import World
    with tempfile.TemporaryDirectory() as tmp:
        sc = edge_scene(tmp)
    rng = np.random.default_rng(11)
    rows = [edge_rows(sc, rng) for _ in range(3)]
    w = World(sc, 3)
    w.state.copy_(torch.from_numpy(np.stack([r[0] for r in rows])))
    w.param.copy_(torch.from_numpy(np.stack([r[1] for r in rows])))
    stats = {}
    for cam in range(sc.hdr['ncam']):
        f, b = render_both(w, cam)
        for e in range(3):
            compare_env(sc, rows[e][0], rows[e][1], cam, tuple(a[e] for a in f), tuple(a[e] for a in b), 'edges cam%d' % cam, stats)
    w.close()
    _report(stats)


def _scene_with_visuals(tmp, nv, cam=(8, 4)):
    static = _urdf(os.path.join(tmp, 'many.urdf'), 'many', [_link('base', _random_visuals(np.random.default_rng(nv), nv, 1.0))], [])
    sb = SceneBuilder()
    sb.add_body('static', static, fixed_base=True)
    eye = np.array([2.0, -1.5, 1.0])
    sb.add_camera(-1, eye, mat_to_quat(look_at(eye, np.zeros(3), 0.2)), cam[0], cam[1], 60.0, 0.05, 8.0)
    return sb.finalize()


def render_smem(nv, static_smem):
    """Shared memory of one render block (render_dyn_smem in csrc/dg_kernels.cu plus the kernel's static buffers)."""
    return static_smem + (max(nv, 1) * 40 + ((nv + 3) & ~3) + (nv + 31) // 32 + 8) * 4


@pytest.mark.gpu
def test_camera_shared_memory_limit():
    """Above 48 KB of static + dynamic shared memory a render needs the opt-in (237 to 299 visual shapes need it for the static
    buffers alone); a scene whose render block exceeds the device's opt-in limit is refused when the world is created."""
    import torch
    from diy_gym_b200.backend import World
    cap = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    static = 10288                                                 # ptxas: t_rgb / t_dep / t_seg / camRp of every instantiation
    nmax = max(nv for nv in range(1, 4000) if render_smem(nv, static) <= cap)
    with tempfile.TemporaryDirectory() as tmp:
        for nv in (237, 299, nmax):
            sc = _scene_with_visuals(tmp, nv)
            w = World(sc, 2)
            f, b = render_both(w, 0)
            ref = cref.render(sc, w.state[0].cpu().numpy().astype(np.float64), w.param[0].cpu().numpy().astype(np.float64), 0)
            assert np.array_equal(f[2][0][~ref['ambiguous']], ref['seg'][~ref['ambiguous']]), nv
            w.close()
        sc = _scene_with_visuals(tmp, nmax + 1)
        with pytest.raises(RuntimeError, match='visual shapes need'):
            World(sc, 2)
    print('camera-kernel shared memory: opt-in limit %d B, largest scene %d visual shapes' % (cap, nmax))


@pytest.mark.gpu
@pytest.mark.parametrize('size', [(7, 3), (100, 60), (160, 90), (88, 64)])
@pytest.mark.parametrize('u8', [False, True])
def test_camera_kernel_writes_nothing_outside_its_images(size, u8):
    """dg_render_seg / dg_render_u8 through the C ABI, each output 256 B into a larger buffer of guard bytes (so it stays 16-byte
    aligned): every pixel is written and every guard byte before and after the images is unchanged."""
    import torch
    from diy_gym_b200.backend import World
    with tempfile.TemporaryDirectory() as tmp:
        sc = synthetic_scene(33, (size, size), tmp)
    N, (wd, hg) = 3, size
    rng = np.random.default_rng(3)
    rows = [random_rows(sc, rng) for _ in range(N)]
    w = World(sc, N)
    w.state.copy_(torch.from_numpy(np.stack([r[0] for r in rows])))
    w.param.copy_(torch.from_numpy(np.stack([r[1] for r in rows])))
    G = 256
    nbytes = (N * hg * wd * 3 * (1 if u8 else 4), N * hg * wd * 4, N * hg * wd * 4)
    bufs = [torch.full((G + nb + G, ), 0x5A, dtype=torch.uint8, device=w.device) for nb in nbytes]
    for cam in (0, 1):
        for bb in bufs:
            bb.fill_(0x5A)
        ptr = [ctypes.c_void_p(bb.data_ptr() + G) for bb in bufs]
        fn = w.L.dg_render_u8 if u8 else w.L.dg_render_seg
        w._check(fn(w._h, cam, ptr[0], ptr[1], ptr[2], w._stream()))
        torch.cuda.synchronize()
        host = [bb.cpu().numpy() for bb in bufs]
        for hb, nb in zip(host, nbytes):
            assert (hb[:G] == 0x5A).all() and (hb[G + nb:] == 0x5A).all(), (size, u8, cam)
        depth, seg = host[1][G:G + nbytes[1]].view(np.float32), host[2][G:G + nbytes[2]].view(np.float32)
        assert (depth < 0).all() and ((seg >= -1) & (seg == np.rint(seg))).all()       # every pixel written
    w.close()
