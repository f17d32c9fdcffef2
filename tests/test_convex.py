"""Convex collision shapes (VERDICT r1 N1; north_star (a)/(b) "primitive/convex"): mesh links are collided as reduced convex hulls
(<= 32 vertices, compiler/mesh.reduced_hull) against boxes and other hulls - vertices of each inside the other, the deepest four
per pair - in the kernels and in the oracle alike.  The reference loads the same meshes as btConvexHullShape (diy_gym/model.py:65)."""
import os

import numpy as np
import pytest
import torch

from diy_gym_b200.assets import resolve_model
from diy_gym_b200.compiler import mesh as cmesh
from diy_gym_b200.compiler.mathutil import quat_to_mat
from diy_gym_b200.compiler.scene import SceneBuilder
from oracle.oracle import OracleWorld
from tests.helpers import golden_mesh, write_mesh

TOUCHING = [2.165, 0.011, 0.699, -1.475, 1.915, 1.938, 0.915, 0.138, -0.472, -0.662, 2.294, -0.915]   # joint angles of the two UR5s of examples/ur_high_5


@pytest.mark.parametrize('rel', ['ur5/meshes/collision/forearm.stl', 'hector_quadrotor/meshes/quadrotor_base.stl', 'jaco/meshes/hand_3finger.dae'])
def test_reduced_hull_approximates_the_mesh_from_inside(rel, tmp_path):
    """The mesh files are not shipped.  The cloud reduced here is made of the mesh vertices kept in tests/golden, points
    inside their hull, and a seeded shell of points up to 1 % of the extent outside its facets, so that the reduction has to
    thin far more than 32 hull vertices as it does on a real mesh.  It goes through the reader of the mesh's format."""
    from scipy.spatial import ConvexHull
    verts, _, _ = golden_mesh(rel)
    rng = np.random.default_rng(7)
    hull = ConvexHull(verts)
    f = rng.integers(0, len(hull.simplices), 400)
    bary = rng.dirichlet(np.ones(3), 400)
    shell = np.einsum('nk,nkd->nd', bary, verts[hull.simplices[f]])
    shell += hull.equations[f, :3] * rng.uniform(0, 0.01 * np.ptp(verts, axis=0).max(), (400, 1))
    inner = rng.dirichlet(np.ones(len(verts)), 200) @ verts
    path = str(tmp_path / os.path.basename(rel))
    write_mesh(path, np.concatenate([verts, shell, inner]))
    v = cmesh.load_vertices(path)
    assert len(v) >= len(verts) + 600 and len(ConvexHull(v).vertices) > 64
    V, P = cmesh.reduced_hull(v)
    assert 4 <= len(V) <= 32 and len(P) <= 64
    assert np.allclose(V.min(axis=0), v.min(axis=0)) and np.allclose(V.max(axis=0), v.max(axis=0))   # the axis extremes are kept
    assert np.allclose(np.linalg.norm(P[:, :3], axis=1), 1.0, atol=1e-9)
    # every reduced vertex is a vertex of the mesh, every one of them satisfies every plane
    assert np.min(np.linalg.norm(v[None, :, :] - V[:, None, :], axis=2), axis=1).max() < 1e-9
    assert (V @ P[:, :3].T - P[:, 3]).max() < 1e-9
    # inner approximation: no mesh vertex sticks out by more than 5 % of the longest extent (rounded parts, 32 vertices)
    out = (v @ P[:, :3].T - P[:, 3]).max(axis=1).max()
    assert 0 <= out < 0.05 * (v.max(0) - v.min(0)).max()


def _hull_world(sc, o, s):
    """world-space vertices of collision shape s from the compiled tables and the oracle's state (independent of the C code)"""
    si, sf, H = sc.sec['SHAPE_I'][s], sc.sec['SHAPE_F'][s], sc.sec['HULL_F']
    V = H[si[4]:si[4] + 3 * si[5]].reshape(-1, 3)
    fs = o.frame_state(int(si[1]))
    R = quat_to_mat(fs['com_quat']) @ quat_to_mat(sf[3:7])
    p = fs['com_pos'] + quat_to_mat(fs['com_quat']) @ sf[0:3]
    return V @ R.T + p


def test_quadrotor_lands_on_the_vertices_of_its_hull():
    sb = SceneBuilder()
    sb.add_body('plane', resolve_model('grass/plane.urdf'))
    sb.add_body('drone', resolve_model('hector_quadrotor/quadrotor.urdf'), xyz=(0, 0, 0.5), mass=4.0)
    sc = sb.finalize()
    hulls = [s for s in range(sc['ns']) if sc.sec['SHAPE_I'][s][5] > 0]
    assert len(hulls) == 1                                         # the quadrotor body mesh
    o = OracleWorld(sc)
    o.env_reset()
    for _ in range(400):
        o.step_physics()
    cs = o.contacts()
    assert len(cs) >= 3
    W = _hull_world(sc, o, hulls[0])
    top = 0.0                                                      # grass/plane.urdf: box 30 x 30 x 10 centred at z = -5
    for c in cs:
        on_drone = c['pa'] if np.linalg.norm(c['n'] - [0, 0, 1]) < 1e-6 else c['pb']
        assert np.abs(np.abs(c['n']) - [0, 0, 1]).max() < 1e-6     # the plane's face normal
        assert np.min(np.linalg.norm(W - on_drone, axis=1)) < 1e-6  # the contact point IS a hull vertex
        assert abs(on_drone[2] - top) < 2e-3                        # resting on the surface
    assert abs(W[:, 2].min() - top) < 2e-3 and np.abs(o.s('S_BVEL', 6)[3:]).max() < 1e-3


def _crossed_arms():
    from diy_gym_b200 import DIYGym
    ex = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'examples', 'ur_high_5', 'ur_high_5.yaml')
    return DIYGym(ex, num_envs=1, compile_only=True).scene


def test_hull_hull_contacts_between_two_arms():
    sc = _crossed_arms()
    o = OracleWorld(sc)
    o.env_reset()
    h = sc.hdr
    # a pose (found by random search) in which links of the two arms interpenetrate by ~3 mm
    o.state[h['S_Q']:h['S_Q'] + 12] = TOUCHING
    o.refresh()
    o.step_physics()
    cs = [c for c in o.contacts()]
    body_of = lambda f: f if f < sc['nb'] else int(sc.sec['LINK_I'][f - sc['nb']][0])
    inter = [c for c in cs if body_of(c['fa']) != body_of(c['fb'])]
    assert len(inter) >= 1, 'the folded arms do not touch: adjust the pose of this test'
    shape_of_frame = {}
    for s in range(sc['ns']):
        shape_of_frame.setdefault(int(sc.sec['SHAPE_I'][s][1]), []).append(s)
    for c in inter:
        assert abs(np.linalg.norm(c['n']) - 1) < 1e-9 and c['dist'] <= 1e-9
        # one of the two points is a hull vertex of its shape, and the points differ by the penetration along the normal
        assert np.allclose(np.asarray(c['pa']) - np.asarray(c['pb']), np.asarray(c['n']) * c['dist'], atol=1e-9)
        hit = False
        for f, pt in ((c['fa'], c['pa']), (c['fb'], c['pb'])):
            for s in shape_of_frame.get(f, []):
                if sc.sec['SHAPE_I'][s][5] > 0 and np.min(np.linalg.norm(_hull_world_pre(sc, o, s) - pt, axis=1)) < 1e-3:
                    hit = True
        assert hit


def _hull_world_pre(sc, o, s):
    return _hull_world(sc, o, s)


def _parity(factory):
    """kernel source against the oracle with hull-hull and hull-box contacts active: one step from identical states"""
    from diy_gym_b200 import DIYGym
    ex = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'examples', 'ur_high_5', 'ur_high_5.yaml')
    env = DIYGym(ex, num_envs=2, device=0, world_factory=factory)
    sc, w, h = env.scene, env.world, env.scene.hdr
    o = OracleWorld(sc)
    o.env_reset()
    o.state[h['S_Q']:h['S_Q'] + 12] = TOUCHING
    o.state[h['S_MTPOS']:h['S_MTPOS'] + 12] = o.state[h['S_Q']:h['S_Q'] + 12]
    o.refresh()
    st = np.stack([o.state, o.state]).astype(np.float32)
    w.state.copy_(torch.from_numpy(st))
    o.state[:] = st[0]
    a = np.zeros((2, sc['n_act']), np.float32)
    w.action.copy_(torch.from_numpy(a))
    w.step()
    o.env_step(a[0].astype(np.float64))
    assert len(o.contacts()) >= 1
    got = w.state[0].cpu().numpy().astype(np.float64)
    nd = sc['nd']
    assert np.allclose(got[h['S_Q']:h['S_Q'] + nd], o.state[h['S_Q']:h['S_Q'] + nd], rtol=1e-4, atol=1e-5)
    assert np.allclose(got[h['S_QD']:h['S_QD'] + nd], o.state[h['S_QD']:h['S_QD'] + nd], rtol=2e-2, atol=2e-2)
    env.close()


def test_hull_contacts_kernel_source_matches_oracle_cpu():
    from tests.emul.world import factory
    _parity(factory(4))


@pytest.mark.gpu
def test_hull_contacts_cuda_matches_oracle():
    _parity(None)
