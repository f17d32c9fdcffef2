"""ctypes wrapper of the CPU emulation of the device code (tests/emul/emul.cpp).  TEST INFRASTRUCTURE: lets the GPU-less
container check the kernel logic (fp32, team phases, ray / dynamics / IK queries) against the fp64 oracle and references."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, '..', '..', 'diy_gym_b200', 'csrc')
_LIB = None


def build(force=False):
    """The emulation library, rebuilt when emul.cpp or any file of the device code is newer.  Written under a name of its own
    and renamed into place, so that test processes running side by side never load a half-written library."""
    so = os.path.join(_HERE, 'libdgemul.so')
    src = os.path.join(_HERE, 'emul.cpp')
    srcs = [src] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
    if force or not os.path.isfile(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        tmp = '%s.%d.tmp' % (so, os.getpid())
        subprocess.check_call(['g++', '-O2', '-fPIC', '-shared', '-std=c++17', '-Wno-unknown-pragmas', '-o', tmp, src])
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        fp, ip, dp, vp, u8 = (ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double),
                              ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint8))
        L.dge_create.restype = vp
        L.dge_create.argtypes = [ip, ctypes.c_int, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.dge_cold_floats.restype = ctypes.c_int
        L.dge_cold_floats.argtypes = [vp]
        L.dge_destroy.argtypes = [vp]
        L.dge_state.restype = fp
        L.dge_state.argtypes = [vp]
        L.dge_param.restype = fp
        L.dge_param.argtypes = [vp]
        L.dge_ws_floats.restype = ctypes.c_int
        L.dge_ws_floats.argtypes = [vp]
        L.dge_set_seed.argtypes = [vp, ctypes.c_uint32, ctypes.c_int]
        L.dge_set_action_mask.argtypes = [vp, u8, ctypes.c_int]
        L.dge_step.argtypes = [vp, fp, fp, fp, u8]
        L.dge_reset.argtypes = [vp, u8, fp, fp, u8]
        L.dge_physics.argtypes = [vp, ctypes.c_int]
        L.dge_observe.argtypes = [vp, fp, fp, u8]
        L.dge_contacts_dropped.restype = ctypes.c_uint
        L.dge_contacts_dropped.argtypes = [vp]
        L.dge_rays.argtypes = [vp, fp, fp, ctypes.c_int, u8]
        L.dge_dynamics.argtypes = [vp, ctypes.c_int, ctypes.c_int, fp, fp, fp, fp, fp, fp, fp, fp, fp, ctypes.c_int]
        L.dge_ik.argtypes = [vp, ctypes.c_int, ctypes.c_int, fp, fp, fp, fp, ctypes.c_int, ctypes.c_float, fp, fp, fp, ctypes.c_int]
        _LIB = L
    return _LIB


def _fp(a):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def _f32(a):
    return None if a is None else np.ascontiguousarray(a, np.float32)


class EmulWorld:
    def __init__(self, scene, n_envs=1, team=1, seed=1234, env_off=0, ws_mode=2):
        L = lib()
        self.scene, self.h, self.n = scene, scene.hdr, n_envs
        ib = np.ascontiguousarray(scene.ibuf, np.int32)
        fb = np.ascontiguousarray(scene.fbuf, np.float64)
        self._w = L.dge_create(ib.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ib.size, fb.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                               fb.size, n_envs, team, ws_mode)
        if not self._w:
            raise RuntimeError('emulation rejected the scene')
        S, P = self.h['S'], self.h['P']
        self.state = np.ctypeslib.as_array(L.dge_state(self._w), shape=(n_envs * S + 1, ))[:n_envs * S].reshape(n_envs, S)
        self.param = np.ctypeslib.as_array(L.dge_param(self._w), shape=(n_envs * P + 1, ))[:n_envs * P].reshape(n_envs, P)
        self.ws_floats = L.dge_ws_floats(self._w)
        self.cold_floats = L.dge_cold_floats(self._w)
        L.dge_set_seed(self._w, seed, env_off)

    def __del__(self):
        if getattr(self, '_w', None):
            lib().dge_destroy(self._w)
            self._w = None

    def s(self, name, n, env=0):
        return self.state[env, self.h[name]:self.h[name] + n]

    def p(self, name, n, env=0):
        return self.param[env, self.h[name]:self.h[name] + n]

    def _outptrs(self):
        h = self.h
        self._o = np.zeros((self.n, max(h['n_obs'], 1)), np.float32)
        self._r = np.zeros((self.n, max(h['n_rew'], 1)), np.float32)
        self._t = np.zeros((self.n, max(h['n_term'], 1)), np.uint8)
        if h['n_obs'] == 0 or h['n_rew'] == 0 or h['n_term'] == 0:
            pass  # zero-width rows: the C side never writes them
        return _fp(self._o), _fp(self._r), self._t.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))

    def _outs(self):
        h = self.h
        return self._o[:, :h['n_obs']], self._r[:, :h['n_rew']], self._t[:, :h['n_term']]

    def step(self, act):
        act = np.ascontiguousarray(act, np.float32).reshape(self.n, -1) if self.h['n_act'] else np.zeros((self.n, 1), np.float32)
        o, r, t = self._outptrs()
        lib().dge_step(self._w, _fp(act), o, r, t)
        return self._outs()

    def observe(self):
        o, r, t = self._outptrs()
        lib().dge_observe(self._w, o, r, t)
        return self._outs()

    def contacts_dropped(self):
        return int(lib().dge_contacts_dropped(self._w))

    def reset(self, mask=None):
        o, r, t = self._outptrs()
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8).ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
        lib().dge_reset(self._w, m, o, r, t)
        return self._outs()

    def physics(self, nsub=None):
        lib().dge_physics(self._w, self.h['substeps'] if nsub is None else nsub)

    # The kernels that read state rows, on explicit rows (numpy, any float dtype) rather than the world's own.
    def rays(self, state, obs=None, mask=None):
        """The ray_sensor ops (dg_ray_kernel) from state rows [n, S] into the ray slices of observation rows [n, n_obs]: in place
        when obs (float32, C-contiguous) is given, else into fresh rows that hold only the rays.  mask: only those environments."""
        h = self.h
        state = np.ascontiguousarray(np.atleast_2d(state), np.float32)
        if obs is None:
            obs = np.zeros((len(state), max(h['n_obs'], 1)), np.float32)
        assert obs.dtype == np.float32 and obs.flags.c_contiguous and state.shape[1] == h['S']
        assert obs.shape[1] >= h['n_obs'] and (obs.shape[1] == max(h['n_obs'], 1) or len(obs) == 1)   # (the C side's row stride: n_obs)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        lib().dge_rays(self._w, _fp(state), _fp(obs), len(state), None if m is None else m.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
        return obs[:, :h['n_obs']]

    def dynamics(self, state, param, body, link=-1, point=(0., 0., 0.), q=None, qd=None, qdd=None, jac=True, mass=True, tau=True):
        """dg_dyn_kernel: (jac [N,6,n], mass [N,n,n], tau [N,n]) as numpy float32 (None where not asked for)."""
        b = self.scene.bodies[body]
        n = b.n_dofs + (6 if b.kind == 2 else 0)
        state, param, point, q, qd, qdd = _f32(state), _f32(param), _f32(point), _f32(q), _f32(qd), _f32(qdd)
        N = len(state)
        outs = [np.zeros((N, 6, n), np.float32) if jac else None, np.zeros((N, n, n), np.float32) if mass else None,
                np.zeros((N, n), np.float32) if tau else None]
        lib().dge_dynamics(self._w, int(body), int(link), _fp(point), _fp(q), _fp(qd), _fp(qdd), *[_fp(o) for o in outs],
                           _fp(state), _fp(param), N)
        return tuple(outs)

    def ik(self, state, body, link, tpos, torn=None, q=None, limits=None, iters=20, threshold=1e-4):
        """dg_ik_kernel: (q [N, n_dof], err [N, 2]) as numpy float32; tpos [N, 3], torn [N, 4], q [N, n_dof], limits [N, 4, n_dof] or
        None."""
        nd, N = self.scene.bodies[body].n_dofs, len(state)
        state, tpos, torn, q, limits = _f32(state), _f32(tpos), _f32(torn), _f32(q), _f32(limits)
        q_out, err = np.zeros((N, nd), np.float32), np.zeros((N, 2), np.float32)
        lib().dge_ik(self._w, int(body), int(link), _fp(tpos), _fp(torn), _fp(q), _fp(limits), int(iters), float(threshold), _fp(q_out),
                     _fp(err), _fp(state), N)
        return q_out, err
