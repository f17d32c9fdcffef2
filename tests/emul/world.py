"""TEST INFRASTRUCTURE: a CPU stand-in with the interface of diy_gym_b200.backend.World, backed by the g++ build
of the device code (tests/emul/emul.cpp) and, for camera images, by the oracle's ray caster.  It lets the
GPU-less container exercise the whole host layer (DIYGym, Model, add-ons); the product never uses it."""
import ctypes

import numpy as np
import torch

from oracle.oracle import OracleWorld
from .emul import EmulWorld, _fp, lib


def _np(t):
    return None if t is None else t.detach().cpu().numpy()


class EmulTorchWorld:
    def __init__(self, scene, n_envs, seed=1234, env_id_offset=0, team=4):
        self.scene, self.n_envs = scene, n_envs
        self.e = EmulWorld(scene, n_envs, team, seed=seed, env_off=env_id_offset)
        h = scene.hdr
        self.n_act, self.n_obs, self.n_rew, self.n_term = h['n_act'], h['n_obs'], h['n_rew'], h['n_term']
        self.state = torch.from_numpy(self.e.state)
        self.param = torch.from_numpy(self.e.param)
        self._a = np.zeros((n_envs, max(self.n_act, 1)), np.float32)
        self._o = np.zeros((n_envs, max(self.n_obs, 1)), np.float32)
        self._r = np.zeros((n_envs, max(self.n_rew, 1)), np.float32)
        self._t = np.zeros((n_envs, max(self.n_term, 1)), np.uint8)
        # the C side indexes rows with the true widths, so these must be exactly [n_envs][width]
        self._a, self._o = self._a[:, :max(self.n_act, 1)], self._o[:, :max(self.n_obs, 1)]
        self.action = torch.from_numpy(self._a)[:, :self.n_act]
        self.obs = torch.from_numpy(self._o)[:, :self.n_obs]
        self.reward = torch.from_numpy(self._r)[:, :self.n_rew]
        self.term = torch.from_numpy(self._t)[:, :self.n_term]
        self.cams = [(int(c[1]), int(c[2])) for c in scene.sec['CAM_I']]
        self.launches = 0
        self._oracle = None

    def _ptrs(self):
        return _fp(self._o), _fp(self._r), self._t.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))

    # step / reset / observe cast the ray_sensor rays afterwards, as the backend's launches do (a reset: the masked environments only)
    def step(self):
        self.launches += 1
        lib().dge_step(self.e._w, _fp(self._a), *self._ptrs())
        self.e.rays(self.e.state, self._o)

    def set_seed(self, seed, env_id_offset=0):
        lib().dge_set_seed(self.e._w, int(seed) & 0xffffffff, int(env_id_offset))

    def observe(self):
        self.launches += 1
        lib().dge_observe(self.e._w, *self._ptrs())
        self.e.rays(self.e.state, self._o)

    def contacts_dropped(self):
        return self.e.contacts_dropped()

    def reset(self, mask=None):
        self.launches += 1
        m = None if mask is None else np.ascontiguousarray(mask.to(torch.uint8).cpu().numpy())
        lib().dge_reset(self.e._w, None if m is None else m.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), *self._ptrs())
        self.e.rays(self.e.state, self._o, m)

    def body_dynamics(self, body, link=-1, point=(0., 0., 0.), q=None, qd=None, qdd=None, jac=False, mass=False, tau=False):
        out = self.e.dynamics(self.e.state, self.e.param, body, link, point, _np(q), _np(qd), _np(qdd), jac, mass, tau)
        return tuple(None if o is None else torch.from_numpy(o) for o in out)

    def body_ik(self, body, link, target_pos, target_orn=None, q=None, limits=None, max_iters=20, threshold=1e-4, err=False):
        q_out, e = self.e.ik(self.e.state, body, link, _np(target_pos), _np(target_orn), _np(q), _np(limits), max_iters, threshold)
        return torch.from_numpy(q_out), torch.from_numpy(e) if err else None

    def render(self, cam=0, seg=False, u8=False):
        if self._oracle is None:
            self._oracle = OracleWorld(self.scene)
        w, hgt = self.cams[cam]
        rgb = np.zeros((self.n_envs, hgt, w, 3), np.float32)
        depth = np.zeros((self.n_envs, hgt, w), np.float32)
        mask = np.zeros((self.n_envs, hgt, w), np.float32)
        for e in range(self.n_envs):
            self._oracle.state[:] = self.e.state[e]
            self._oracle.param[:] = self.e.param[e]
            out = self._oracle.render(cam, seg=seg)
            rgb[e], depth[e] = out[0], out[1]
            if seg:
                mask[e] = out[2]
        if u8:   # round(255 c), as dg_render_u8
            rgb = np.rint(np.clip(rgb, 0.0, 1.0) * 255.0).astype(np.uint8)
        return (torch.from_numpy(rgb), torch.from_numpy(depth)) + ((torch.from_numpy(mask), ) if seg else ())

    def set_action_mask(self, enabled):
        m = np.ascontiguousarray(enabled, np.uint8)
        lib().dge_set_action_mask(self.e._w, m.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), m.size)

    def close(self):
        pass


def factory(team=4):
    return lambda scene, n, seed, off: EmulTorchWorld(scene, n, seed, off, team)
