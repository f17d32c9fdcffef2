"""ctypes wrapper of the CPU build of the ray_sensor routines (tests/emul/ray_emul.cpp), and a stand-in world for the host layer
that runs them after every step / reset / observe of the step-code emulation, as the CUDA backend launches dg_ray_kernel.
TEST INFRASTRUCTURE: the product never uses it."""
import ctypes
import os
import subprocess

import numpy as np

from .world import EmulTorchWorld

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, '..', '..', 'diy_gym_b200', 'csrc')
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, 'libdgrayemul.so')
    srcs = [os.path.join(_HERE, 'ray_emul.cpp')] + [os.path.join(_CSRC, f) for f in ('dg_ray.cuh', 'dg_env.cuh', 'dg_math.cuh', 'dg_scene.h',
                                                                                       'scene_sections.h')]
    if force or not os.path.isfile(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(['g++', '-O2', '-fPIC', '-shared', '-std=c++17', '-Wno-unknown-pragmas', '-o', so, srcs[0]])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        fp, vp, u8 = ctypes.POINTER(ctypes.c_float), ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint8)
        L.dgr_create.restype = vp
        L.dgr_create.argtypes = [ctypes.POINTER(ctypes.c_int32), ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.c_int]
        L.dgr_destroy.argtypes = [vp]
        L.dgr_rays.argtypes = [vp, fp, fp, ctypes.c_int, u8]
        _LIB = L
    return _LIB


class RayCaster:
    """The fp32 ray_sensor routines of one compiled scene, cast from state rows into observation rows."""
    def __init__(self, scene):
        self.scene = scene
        ib = np.ascontiguousarray(scene.ibuf, np.int32)
        fb = np.ascontiguousarray(scene.fbuf, np.float64)
        self._w = lib().dgr_create(ib.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ib.size,
                                   fb.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), fb.size)
        if not self._w:
            raise RuntimeError('ray emulation rejected the scene')

    def __del__(self):
        if getattr(self, '_w', None):
            lib().dgr_destroy(self._w)
            self._w = None

    def cast(self, state, obs, mask=None):
        """state [n, S] and obs [n, n_obs] float32 C-contiguous arrays; the ray slices of obs are written in place."""
        h = self.scene.hdr
        assert state.dtype == np.float32 and obs.dtype == np.float32 and state.flags.c_contiguous and obs.flags.c_contiguous
        assert state.shape[1] == h['S'] and obs.shape[1] >= h['n_obs'] and (obs.shape[1] == h['n_obs'] or len(obs) == 1)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        fp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        lib().dgr_rays(self._w, fp(state), fp(obs), len(state), None if m is None else m.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
        return obs

    def rays(self, state):
        """Observation rows [n, n_obs] holding only the ray slices, from state rows [n, S] (any float dtype)."""
        st = np.ascontiguousarray(np.atleast_2d(state), np.float32)
        return self.cast(st, np.zeros((len(st), max(self.scene.hdr['n_obs'], 1)), np.float32))[:, :self.scene.hdr['n_obs']]


class RayEmulTorchWorld(EmulTorchWorld):
    """EmulTorchWorld plus the ray_sensor ops after every step / reset (masked environments only) / observe."""
    def __init__(self, scene, n_envs, seed=1234, env_id_offset=0, team=4):
        super().__init__(scene, n_envs, seed, env_id_offset, team)
        self._rays = RayCaster(scene)

    def step(self):
        super().step()
        self._rays.cast(self.e.state, self._o)

    def observe(self):
        super().observe()
        self._rays.cast(self.e.state, self._o)

    def reset(self, mask=None):
        super().reset(mask)
        self._rays.cast(self.e.state, self._o, None if mask is None else self._m)


def factory(team=4):
    return lambda scene, n, seed, off: RayEmulTorchWorld(scene, n, seed, off, team)
