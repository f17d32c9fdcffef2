"""ctypes wrapper of the CPU build of the dynamics-query routines (tests/emul/dyn_emul.cpp), and a stand-in world for the host
layer that answers `body_dynamics` with them, as the CUDA backend launches dg_dyn_kernel.  TEST INFRASTRUCTURE: the product never
uses it."""
import ctypes
import os
import subprocess

import numpy as np
import torch

from .world import EmulTorchWorld

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, '..', '..', 'diy_gym_b200', 'csrc')
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, 'libdgdynemul.so')
    srcs = [os.path.join(_HERE, 'dyn_emul.cpp')] + [os.path.join(_CSRC, f) for f in ('dg_dyn.cuh', 'dg_math.cuh', 'dg_scene.h', 'scene_sections.h')]
    if force or not os.path.isfile(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(['g++', '-O2', '-fPIC', '-shared', '-std=c++17', '-Wno-unknown-pragmas', '-o', so, srcs[0]])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        fp, vp = ctypes.POINTER(ctypes.c_float), ctypes.c_void_p
        L.dgd_create.restype = vp
        L.dgd_create.argtypes = [ctypes.POINTER(ctypes.c_int32), ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.c_int]
        L.dgd_destroy.argtypes = [vp]
        L.dgd_dynamics.argtypes = [vp, ctypes.c_int, ctypes.c_int, fp, fp, fp, fp, fp, fp, fp, fp, fp, ctypes.c_int]
        _LIB = L
    return _LIB


class DynEmul:
    """The fp32 dynamics routines of one compiled scene, evaluated from state / parameter rows (numpy float32, C-contiguous)."""
    def __init__(self, scene):
        self.scene = scene
        ib = np.ascontiguousarray(scene.ibuf, np.int32)
        fb = np.ascontiguousarray(scene.fbuf, np.float64)
        self._w = lib().dgd_create(ib.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ib.size,
                                   fb.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), fb.size)
        if not self._w:
            raise RuntimeError('dynamics emulation rejected the scene')

    def __del__(self):
        if getattr(self, '_w', None):
            lib().dgd_destroy(self._w)
            self._w = None

    def dynamics(self, state, param, body, link=-1, point=(0., 0., 0.), q=None, qd=None, qdd=None, jac=True, mass=True, tau=True):
        """(jac [N,6,n], mass [N,n,n], tau [N,n]) as numpy float32 (None where not asked for)."""
        b = self.scene.bodies[body]
        n = b.n_dofs + (6 if b.kind == 2 else 0)
        N = len(state)
        f32 = lambda a: None if a is None else np.ascontiguousarray(a, np.float32)
        state, param, q, qd, qdd = f32(state), f32(param), f32(q), f32(qd), f32(qdd)
        outs = [np.zeros((N, 6, n), np.float32) if jac else None, np.zeros((N, n, n), np.float32) if mass else None,
                np.zeros((N, n), np.float32) if tau else None]
        fp = lambda a: None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        pt = np.ascontiguousarray(point, np.float32)
        lib().dgd_dynamics(self._w, int(body), int(link), fp(pt), fp(q), fp(qd), fp(qdd), *[fp(o) for o in outs], fp(state), fp(param), N)
        return tuple(outs)


class DynEmulTorchWorld(EmulTorchWorld):
    """EmulTorchWorld plus `body_dynamics` (the interface of backend.World) from the g++ build of dg_dyn.cuh."""
    def __init__(self, scene, n_envs, seed=1234, env_id_offset=0, team=4):
        super().__init__(scene, n_envs, seed, env_id_offset, team)
        self._dyn = DynEmul(scene)

    def body_dynamics(self, body, link=-1, point=(0., 0., 0.), q=None, qd=None, qdd=None, jac=False, mass=False, tau=False):
        np_ = lambda t: None if t is None else t.detach().cpu().numpy()
        out = self._dyn.dynamics(self.e.state, self.e.param, body, link, point, np_(q), np_(qd), np_(qdd), jac, mass, tau)
        return tuple(None if o is None else torch.from_numpy(o) for o in out)


def factory(team=4):
    return lambda scene, n, seed, off: DynEmulTorchWorld(scene, n, seed, off, team)
