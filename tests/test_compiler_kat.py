"""Known-answer tests of the COMPILER products that the kernels and the oracle both consume (VERDICT r1 weak 4: the oracle is
not independent of diy_gym_b200/compiler - a wrong inertia rule, proxy fit or joint frame would be invisible to every parity
test).  Each test recomputes the expected value from the source asset with nothing but the standard library / numpy:
inertia diagonals from closed forms on the URDF's own <geometry>, mesh bounding boxes from the raw vertices against the table of
SURVEY Appendix B.3, getJointInfo fields from the URDF XML."""
import os
import struct
import xml.etree.ElementTree as ET

import numpy as np
import pytest

from diy_gym_b200.assets import resolve_model
from diy_gym_b200.compiler import mesh as cmesh
from diy_gym_b200.compiler.scene import SceneBuilder
from diy_gym_b200.compiler.urdf import compile_urdf, inertia_from_rule
from tests.helpers import golden_mesh, write_mesh

DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'diy_gym_b200', 'data')


def _urdf_path(rel):
    for root, _, files in os.walk(DATA):
        if os.path.basename(rel) in files and root.replace('\\', '/').endswith(os.path.dirname(rel)):
            return os.path.join(root, os.path.basename(rel))
    pytest.skip('asset %s not vendored' % rel)


def _closed_form(geom, mass):
    """Inertia diagonal of a solid primitive about its centre, textbook formulas on the XML's own numbers."""
    if geom.find('box') is not None:
        lx, ly, lz = [float(v) for v in geom.find('box').get('size').split()]
        return mass / 12.0 * np.array([ly * ly + lz * lz, lx * lx + lz * lz, lx * lx + ly * ly])
    if geom.find('sphere') is not None:
        r = float(geom.find('sphere').get('radius'))
        return np.full(3, 0.4 * mass * r * r)
    if geom.find('cylinder') is not None:
        r, l = float(geom.find('cylinder').get('radius')), float(geom.find('cylinder').get('length'))
        return np.array([mass * (3 * r * r + l * l) / 12.0] * 2 + [0.5 * mass * r * r])
    return None


@pytest.mark.parametrize('rel', ['standin/r2d2.urdf', 'standin/sphere2.urdf'])
def test_inertia_of_single_primitive_links_is_the_closed_form(rel):
    """Links whose only collision shape is a primitive coincident with the inertial frame: Bullet's calculateLocalInertia of
    that primitive (SURVEY App. A.1) = the textbook formula; the XML <inertia> is ignored."""
    path = resolve_model(os.path.basename(rel)) if not os.path.isfile(os.path.join(DATA, rel)) else None
    desc = path if isinstance(path, dict) else compile_urdf(os.path.join(DATA, rel))
    root = ET.parse(os.path.join(DATA, rel)).getroot()
    checked = 0
    for le in root.findall('link'):
        cols, inertial = le.findall('collision'), le.find('inertial')
        if len(cols) != 1 or inertial is None or inertial.find('mass') is None:
            continue
        mass = float(inertial.find('mass').get('value'))
        want = _closed_form(cols[0].find('geometry'), mass)
        def org(e):
            o = e.find('origin')
            f = lambda t: [float(v) for v in (o.get(t, '0 0 0') if o is not None else '0 0 0').split()]
            return f('xyz'), f('rpy')
        (cx, cr), (ix, ir) = org(cols[0]), org(inertial)
        if want is None or mass <= 0 or cx != ix or cr != [0, 0, 0] or ir != [0, 0, 0]:
            continue
        link = next(l for l in desc['links'] if l['name'] == le.get('name'))
        got = inertia_from_rule(link['inertia_rule'], mass, 1.0, link['inertia_xml'])
        assert np.allclose(got, want, rtol=1e-9), (le.get('name'), got, want)
        checked += 1
    assert checked >= 1, 'no single-primitive link in %s' % rel


def _stl_vertices(path):
    with open(path, 'rb') as f:
        f.read(80)
        n = struct.unpack('<I', f.read(4))[0]
        rec = np.frombuffer(f.read(50 * n), dtype=np.dtype([('n', '<f4', 3), ('v', '<f4', 9), ('a', '<u2')]))
    return rec['v'].reshape(-1, 3).astype(np.float64)


# SURVEY Appendix B.3: AABB of the UR5 collision meshes and of the quadrotor body, metres
B3 = {'ur5/meshes/collision/base.stl': ((-0.0736, -0.110, -0.003), (0.0736, 0.0736, 0.021)),
      'ur5/meshes/collision/upperarm.stl': ((-0.0599, -0.0652, -0.0597), (0.0595, 0.0686, 0.4849)),
      'ur5/meshes/collision/forearm.stl': ((-0.0579, -0.0572, -0.058), (0.0585, 0.0545, 0.4313)),
      'ur5/meshes/collision/wrist3.stl': ((-0.0375, 0.0473, -0.0375), (0.0375, 0.0818, 0.043)),
      'hector_quadrotor/meshes/quadrotor_base.stl': ((-0.3956, -0.3956, -0.1825), (0.3956, 0.3956, 0.040))}


@pytest.mark.parametrize('rel', sorted(B3))
def test_mesh_reader_and_proxy_fit_against_the_survey_table(rel, tmp_path):
    """The compiler's mesh reader gives the bounding box SURVEY B.3 lists, and the fitted collision proxy (capsule / box: meshes
    are not collided as hulls yet, DESIGN.md section 7) stays inside that box inflated by 15 % and covers at least 60 % of its
    longest extent.  The mesh files are not shipped: the test writes the vertices of the mesh kept in tests/golden (its
    extreme vertices along each axis among them, so the same bounding box) as a binary STL and reads that.  fit_proxy
    depends on nothing but the bounding box, so it fits the same proxy as to the whole mesh: the one the descriptor holds."""
    verts, box_lo, box_hi = golden_mesh(rel)
    path = str(tmp_path / os.path.basename(rel))
    write_mesh(path, verts)
    v = cmesh.load_vertices(path)
    assert np.allclose(v, _stl_vertices(path))                               # the reader against an independent STL parse
    assert np.allclose(v[:len(verts)], verts, rtol=1e-6, atol=1e-7)          # float32 round trip
    lo, hi = np.array(B3[rel][0]), np.array(B3[rel][1])
    assert np.allclose(v.min(axis=0), lo, atol=2e-3) and np.allclose(v.max(axis=0), hi, atol=2e-3)
    assert np.allclose(v.min(axis=0), box_lo, atol=1e-7) and np.allclose(v.max(axis=0), box_hi, atol=1e-7)
    fit = cmesh.fit_proxy(v)
    model = 'ur5/ur5_robot.urdf' if rel.startswith('ur5/') else 'hector_quadrotor/quadrotor.urdf'
    col = next(c for l in resolve_model(model)['links'] for c in l['collisions'] if c.get('mesh') == os.path.basename(rel))
    assert fit['type'] == col['type'] and np.allclose(fit['dims'], col['dims'][:len(fit['dims'])], atol=1e-7)
    c, half = np.array(fit['center']), np.array(fit['half'])
    ext = hi - lo
    assert np.all(c - half >= lo - 0.15 * ext.max()) and np.all(c + half <= hi + 0.15 * ext.max())
    assert 2 * half.max() >= 0.6 * ext.max()


def test_joint_info_fields_follow_the_urdf():
    """getJointInfo field order as the add-ons index it ([1] name, [2] type, [3] qIndex, [6] damping, [7] friction, [8] lower,
    [9] upper, [10] max force, [11] max velocity, [13] axis) against the UR5 XML (SURVEY App. B.1: effort 150/150/150/28/28/28,
    limits +-2 pi except the elbow's +-pi)."""
    sb = SceneBuilder()
    b = sb.add_body('ur5', resolve_model('ur5/ur5_robot.urdf'))
    sb.finalize()
    names = b.joint_names()
    movable = b.movable_joints()
    assert [names[i] for i in movable] == ['shoulder_pan_joint', 'shoulder_lift_joint', 'elbow_joint', 'wrist_1_joint', 'wrist_2_joint', 'wrist_3_joint']
    assert movable == [1, 2, 3, 4, 5, 6] and names[7] == 'ee_fixed_joint'
    infos = [b.joint_info(i) for i in movable]
    assert [i['max_force'] for i in infos] == [150.0, 150.0, 150.0, 28.0, 28.0, 28.0]
    assert np.allclose([i['max_velocity'] for i in infos], [3.15, 3.15, 3.15, 3.2, 3.2, 3.2])
    assert np.allclose([i['lower'] for i in infos], [-2 * np.pi, -2 * np.pi, -np.pi, -2 * np.pi, -2 * np.pi, -2 * np.pi], atol=1e-4)
    assert np.allclose([i['upper'] for i in infos], [2 * np.pi, 2 * np.pi, np.pi, 2 * np.pi, 2 * np.pi, 2 * np.pi], atol=1e-4)
    assert all(i['damping'] == 0.0 for i in infos)
    axes = [tuple(float(v) for v in np.round(b.links[i + 1]['joint']['axis'], 6)) for i in movable]
    assert axes == [(0, 0, 1), (0, 1, 0), (0, 1, 0), (0, 1, 0), (0, 0, 1), (0, 1, 0)]
