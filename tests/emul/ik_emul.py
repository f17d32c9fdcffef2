"""ctypes wrapper of the CPU build of the inverse-kinematics query (tests/emul/ik_emul.cpp), and a stand-in world for the host
layer that answers `body_ik` with it, as the CUDA backend launches dg_ik_kernel.  TEST INFRASTRUCTURE: the product never uses
it."""
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
    so = os.path.join(_HERE, 'libdgikemul.so')
    srcs = [os.path.join(_HERE, 'ik_emul.cpp')] + [os.path.join(_CSRC, f) for f in ('dg_ik.cuh', 'dg_env.cuh', 'dg_math.cuh', 'dg_scene.h', 'scene_sections.h')]
    if force or not os.path.isfile(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(['g++', '-O2', '-fPIC', '-shared', '-std=c++17', '-Wno-unknown-pragmas', '-o', so, srcs[0]])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        fp, vp = ctypes.POINTER(ctypes.c_float), ctypes.c_void_p
        L.dgi_create.restype = vp
        L.dgi_create.argtypes = [ctypes.POINTER(ctypes.c_int32), ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.c_int]
        L.dgi_destroy.argtypes = [vp]
        L.dgi_ik.argtypes = [vp, ctypes.c_int, ctypes.c_int, fp, fp, fp, fp, ctypes.c_int, ctypes.c_float, fp, fp, fp, ctypes.c_int]
        _LIB = L
    return _LIB


class IkEmul:
    """The fp32 IK query of one compiled scene, evaluated from state rows (numpy float32, C-contiguous)."""
    def __init__(self, scene, team=4):
        self.scene = scene
        ib = np.ascontiguousarray(scene.ibuf, np.int32)
        fb = np.ascontiguousarray(scene.fbuf, np.float64)
        self._w = lib().dgi_create(ib.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ib.size,
                                   fb.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), fb.size, int(team))
        if not self._w:
            raise RuntimeError('IK emulation rejected the scene')

    def __del__(self):
        if getattr(self, '_w', None):
            lib().dgi_destroy(self._w)
            self._w = None

    def ik(self, state, body, link, tpos, torn=None, q=None, limits=None, iters=20, threshold=1e-4):
        """(q [N, n_dof], err [N, 2]) as numpy float32; tpos [N, 3], torn [N, 4], q [N, n_dof], limits [N, 4, n_dof] or None."""
        nd, N = self.scene.bodies[body].n_dofs, len(state)
        f32 = lambda a: None if a is None else np.ascontiguousarray(a, np.float32)
        state, tpos, torn, q, limits = f32(state), f32(tpos), f32(torn), f32(q), f32(limits)
        q_out, err = np.zeros((N, nd), np.float32), np.zeros((N, 2), np.float32)
        fp = lambda a: None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        lib().dgi_ik(self._w, int(body), int(link), fp(tpos), fp(torn), fp(q), fp(limits), int(iters), float(threshold), fp(q_out),
                     fp(err), fp(state), N)
        return q_out, err


class IkEmulTorchWorld(EmulTorchWorld):
    """EmulTorchWorld plus `body_ik` (the interface of backend.World) from the g++ build of dg_ik.cuh."""
    def __init__(self, scene, n_envs, seed=1234, env_id_offset=0, team=4):
        super().__init__(scene, n_envs, seed, env_id_offset, team)
        self._ik = IkEmul(scene, team)

    def body_ik(self, body, link, target_pos, target_orn=None, q=None, limits=None, max_iters=20, threshold=1e-4, err=False):
        np_ = lambda t: None if t is None else t.detach().cpu().numpy()
        q_out, e = self._ik.ik(self.e.state, body, link, np_(target_pos), np_(target_orn), np_(q), np_(limits), max_iters, threshold)
        return torch.from_numpy(q_out), torch.from_numpy(e) if err else None


def factory(team=4):
    return lambda scene, n, seed, off: IkEmulTorchWorld(scene, n, seed, off, team)
