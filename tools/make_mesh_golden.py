"""Writes tests/golden/mesh_vertices.npz: for each source mesh the compiler tests need, the mesh's axis-aligned bounding box
and the vertices of its reduced convex hull, both in the mesh's own frame.

The mesh files themselves are not shipped.  When the model descriptors in diy_gym_b200/data/compiled/ were compiled from
them, each one kept the bounding box of the mesh and its reduced hull (compiler/mesh.reduced_hull: a subset of the
mesh's vertices that includes the extreme ones along each axis).  This script maps those hull vertices back from the
descriptor's shape frame into the mesh frame and freezes them, so that the tests keep their data if the descriptors are
recompiled.  Usage: python tools/make_mesh_golden.py"""
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, ROOT)
from diy_gym_b200.assets import resolve_model  # noqa: E402
from diy_gym_b200.compiler.mathutil import quat_to_mat  # noqa: E402

# mesh -> a model that references it (every one of them sits at the identity <origin> of its link)
MESHES = {'ur5/meshes/collision/base.stl': 'ur5/ur5_robot.urdf', 'ur5/meshes/collision/upperarm.stl': 'ur5/ur5_robot.urdf',
          'ur5/meshes/collision/forearm.stl': 'ur5/ur5_robot.urdf', 'ur5/meshes/collision/wrist3.stl': 'ur5/ur5_robot.urdf',
          'hector_quadrotor/meshes/quadrotor_base.stl': 'hector_quadrotor/quadrotor.urdf',
          'jaco/meshes/hand_3finger.dae': 'jaco/j2s7s300_standalone.urdf'}


def key(rel):
    return os.path.splitext(os.path.basename(rel))[0]


def main():
    out = {}
    for rel, urdf in MESHES.items():
        col = next(c for l in resolve_model(urdf)['links'] for c in l['collisions'] if c.get('mesh') == os.path.basename(rel))
        a = col['aabb']
        assert a['quat'] == [0.0, 0.0, 0.0, 1.0], rel
        verts = np.asarray(col['hull']['verts']) @ quat_to_mat(np.asarray(col['quat'])).T + np.asarray(col['xyz'])
        lo, hi = np.asarray(a['xyz']) - a['half'], np.asarray(a['xyz']) + a['half']
        assert np.allclose(verts.min(0), lo, atol=1e-9) and np.allclose(verts.max(0), hi, atol=1e-9), rel
        out['verts_' + key(rel)], out['lo_' + key(rel)], out['hi_' + key(rel)] = verts, lo, hi
    np.savez_compressed(os.path.join(ROOT, 'tests', 'golden', 'mesh_vertices.npz'), **out)


if __name__ == '__main__':
    main()
