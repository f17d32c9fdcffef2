"""ctypes binding of the C ABI (include/diygym_b200.h) + the torch-owned device buffers of one world.

There is no CPU fallback: a missing library or a missing CUDA device raises.  PyTorch is used for device
memory and streams only; the arithmetic is in csrc/dg_kernels.cu.
"""
import ctypes
import os

import numpy as np
import torch

from .build import LIB

_lib = None


class DgBufferTable(ctypes.Structure):
    _fields_ = [('state', ctypes.c_void_p), ('param', ctypes.c_void_p), ('action', ctypes.c_void_p), ('obs', ctypes.c_void_p),
                ('reward', ctypes.c_void_p), ('term', ctypes.c_void_p)]


DYN_MAX_N = 64   # DG_DYN_MAX_N of include/diygym_b200.h: largest number of generalized coordinates dg_body_dynamics accepts
IK_MAX_ND = 64   # DG_IK_MAX_ND of include/diygym_b200.h: largest number of DoF dg_body_ik accepts

Q = dict(STATE_SIZE=0, PARAM_SIZE=1, N_ACT=2, N_OBS=3, N_REW=4, N_TERM=5, N_ENVS=6, TEAM=7, BLOCK_THREADS=8, GRID_BLOCKS=9,
         SMEM_BYTES=10, WS_FLOATS=11, N_CAMERAS=12, LAUNCHES=13, RS_ASHARED=14, SOLVER=15, MAX_CONTACTS=16, CONTACTS_DROPPED=17, SPLIT=18)


def load_library():
    """dlopen libdiygym_b200.so (built in-tree by `python -m diy_gym_b200.build`); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB):
        raise RuntimeError('libdiygym_b200.so is missing: run `python -m diy_gym_b200.build` (there is no CPU fallback)')
    L = ctypes.CDLL(LIB)
    vp, ip, dp = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double)
    L.dg_world_create.restype = ctypes.c_int
    L.dg_world_create.argtypes = [ip, ctypes.c_int, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(vp)]
    L.dg_world_destroy.restype = None
    L.dg_world_destroy.argtypes = [vp]
    L.dg_last_error.restype = ctypes.c_char_p
    L.dg_last_error.argtypes = [vp]
    L.dg_query.restype = ctypes.c_int64
    L.dg_query.argtypes = [vp, ctypes.c_int]
    L.dg_bind_buffers.restype = ctypes.c_int
    L.dg_bind_buffers.argtypes = [vp, ctypes.POINTER(DgBufferTable)]
    L.dg_set_seed.restype = ctypes.c_int
    L.dg_set_seed.argtypes = [vp, ctypes.c_uint32, ctypes.c_int]
    for f in ('dg_init_state', 'dg_step', 'dg_observe'):
        getattr(L, f).restype = ctypes.c_int
        getattr(L, f).argtypes = [vp, vp]
    L.dg_reset.restype = ctypes.c_int
    L.dg_reset.argtypes = [vp, vp, vp]
    L.dg_render.restype = ctypes.c_int
    L.dg_render.argtypes = [vp, ctypes.c_int, vp, vp, vp]
    L.dg_render_seg.restype = ctypes.c_int
    L.dg_render_seg.argtypes = [vp, ctypes.c_int, vp, vp, vp, vp]
    L.dg_render_u8.restype = ctypes.c_int
    L.dg_render_u8.argtypes = [vp, ctypes.c_int, vp, vp, vp, vp]
    L.dg_set_action_mask.restype = ctypes.c_int
    L.dg_set_action_mask.argtypes = [vp, ctypes.POINTER(ctypes.c_uint8), ctypes.c_int]
    L.dg_step_host.restype = ctypes.c_int
    L.dg_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    L.dg_debug_phase_cycles.restype = ctypes.c_int
    L.dg_debug_phase_cycles.argtypes = [vp, ctypes.c_int]
    L.dg_debug_read.restype = ctypes.c_int
    L.dg_debug_read.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64), ctypes.c_int]
    L.dg_body_dynamics.restype = ctypes.c_int
    L.dg_body_dynamics.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float), vp, vp, vp, vp, vp, vp, vp]
    L.dg_body_ik.restype = ctypes.c_int
    L.dg_body_ik.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int, ctypes.c_float, vp, vp, vp]
    L.dg_measure_fp32_peak.restype = ctypes.c_int
    L.dg_measure_fp32_peak.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    _lib = L
    return L


def measure_fp32_peak(device=0):
    """Non-tensor FP32 FMA rate of the device in TFLOP/s (measured by an FMA micro-kernel)."""
    out = ctypes.c_double(0.0)
    rc = load_library().dg_measure_fp32_peak(int(device), ctypes.byref(out))
    if rc != 0:
        raise RuntimeError('dg_measure_fp32_peak failed: %d' % rc)
    return out.value


class World:
    """N lock-stepped environments of one compiled scene on one GPU."""
    def __init__(self, scene, n_envs, device=0, team=0, seed=1234, env_id_offset=0):
        if not torch.cuda.is_available():
            raise RuntimeError('diy_gym_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
        L = load_library()
        self.L, self.scene, self.n_envs = L, scene, int(n_envs)
        self.device = torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)
        ib = np.ascontiguousarray(scene.ibuf, np.int32)
        fb = np.ascontiguousarray(scene.fbuf, np.float64)
        h = ctypes.c_void_p()
        rc = L.dg_world_create(ib.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ib.size, fb.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                               fb.size, self.n_envs, self.device.index, int(team), ctypes.byref(h))
        if rc != 0:
            raise RuntimeError('dg_world_create failed (%d): %s' % (rc, L.dg_last_error(None).decode()))
        self._h = h
        q = lambda k: int(L.dg_query(h, Q[k]))
        self.S, self.P, self.n_act, self.n_obs, self.n_rew, self.n_term = q('STATE_SIZE'), q('PARAM_SIZE'), q('N_ACT'), q('N_OBS'), q('N_REW'), q('N_TERM')
        self.team, self.block_threads, self.grid_blocks, self.smem_bytes, self.ws_floats = q('TEAM'), q('BLOCK_THREADS'), q('GRID_BLOCKS'), q('SMEM_BYTES'), q('WS_FLOATS')
        N, dev = self.n_envs, self.device
        self.state = torch.zeros((N, self.S), dtype=torch.float32, device=dev)
        self.param = torch.zeros((N, self.P), dtype=torch.float32, device=dev)
        self.action = torch.zeros((N, max(self.n_act, 1)), dtype=torch.float32, device=dev)[:, :self.n_act].contiguous() if self.n_act else torch.zeros((N, 0), dtype=torch.float32, device=dev)
        self.obs = torch.zeros((N, self.n_obs), dtype=torch.float32, device=dev)
        self.reward = torch.zeros((N, self.n_rew), dtype=torch.float32, device=dev)
        self.term = torch.zeros((N, self.n_term), dtype=torch.uint8, device=dev)
        self._keep = [torch.zeros(4, device=dev) for _ in range(4)]   # non-null stand-ins for zero-width buffers
        ptr = lambda t, i: t.data_ptr() if t.numel() else self._keep[i].data_ptr()
        tab = DgBufferTable(self.state.data_ptr(), self.param.data_ptr(), ptr(self.action, 0), ptr(self.obs, 1), ptr(self.reward, 2), ptr(self.term, 3))
        self._check(L.dg_bind_buffers(h, ctypes.byref(tab)))
        self._check(L.dg_set_seed(h, int(seed) & 0xffffffff, int(env_id_offset)))
        self._check(L.dg_init_state(h, self._stream()))
        self.cams = [(int(c[1]), int(c[2])) for c in scene.sec['CAM_I']]
        self._img = {}

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError('diygym_b200 error %d: %s' % (rc, self.L.dg_last_error(self._h).decode()))

    def close(self):
        if getattr(self, '_h', None):
            torch.cuda.synchronize(self.device)
            self.L.dg_world_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def split(self):
        """True while a step runs as stage launches around the contact-sweep kernel (adaptive: see dg_kernels.cu)."""
        return bool(self.L.dg_query(self._h, Q['SPLIT']))

    @property
    def launches(self):
        return int(self.L.dg_query(self._h, Q['LAUNCHES']))

    def step(self):
        self._check(self.L.dg_step(self._h, self._stream()))

    def set_seed(self, seed, env_id_offset=0):
        self._check(self.L.dg_set_seed(self._h, int(seed) & 0xffffffff, int(env_id_offset)))

    def observe(self):
        """Outputs (obs / reward / term) from the state rows as they are: link cache refresh + every sensor op, no physics."""
        self._check(self.L.dg_observe(self._h, self._stream()))

    def contacts_dropped(self):
        """Contacts lost to the `max_contacts` capacity since creation (synchronises)."""
        return int(self.L.dg_query(self._h, Q['CONTACTS_DROPPED']))

    def reset(self, mask=None):
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        self._check(self.L.dg_reset(self._h, ctypes.c_void_p(mask.data_ptr()) if mask is not None else None, self._stream()))

    def set_action_mask(self, enabled):
        m = np.ascontiguousarray(enabled, np.uint8)
        self._check(self.L.dg_set_action_mask(self._h, m.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), m.size))

    def render(self, cam=0, seg=False, u8=False):
        """Camera `cam` of every environment: (rgb [N, H, W, 3], depth [N, H, W][, mask [N, H, W]]) - views of buffers the next
        render overwrites.  u8: the colour image as bytes round(255 c) (what the reference divides by 255, camera.py:76-78)."""
        w, hgt = self.cams[cam]
        key = ('u8', cam) if u8 else cam
        if key not in self._img:
            self._img[key] = (torch.empty((self.n_envs, hgt, w, 3), dtype=torch.uint8 if u8 else torch.float32, device=self.device),
                              torch.empty((self.n_envs, hgt, w), dtype=torch.float32, device=self.device))
        rgb, depth = self._img[key]
        mask = None
        if seg:
            if ('seg', cam) not in self._img:
                self._img[('seg', cam)] = torch.empty((self.n_envs, hgt, w), dtype=torch.float32, device=self.device)
            mask = self._img[('seg', cam)]
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        if u8:
            self._check(self.L.dg_render_u8(self._h, cam, p(rgb), p(depth), p(mask), self._stream()))
        elif seg:
            self._check(self.L.dg_render_seg(self._h, cam, p(rgb), p(depth), p(mask), self._stream()))
        else:
            self._check(self.L.dg_render(self._h, cam, p(rgb), p(depth), self._stream()))
        return (rgb, depth, mask) if seg else (rgb, depth)

    def step_host(self, action_host, obs_host, reward_host, term_host):
        """Host-buffer step: numpy (ideally pinned) in, numpy out, synchronous."""
        p = lambda a: ctypes.c_void_p(a.ctypes.data) if a is not None and a.size else None
        self._check(self.L.dg_step_host(self._h, p(action_host), p(obs_host), p(reward_host), p(term_host), self._stream()))

    def body_dynamics(self, body, link=-1, point=(0., 0., 0.), q=None, qd=None, qdd=None, jac=False, mass=False, tau=False):
        """Jacobian [N, 6, n] (linear rows first), mass matrix [N, n, n] and inverse dynamics [N, n] of body `body` (dg_body_dynamics):
        new tensors, None where not asked for.  q [N, n_dof], qd / qdd [N, n]: contiguous float32 tensors on this world's device or
        None (the state row's q, the state row's velocities, zero).  Asynchronous on the current stream."""
        b = self.scene.bodies[body]
        n, N, dev = b.n_dofs + (6 if b.kind == 2 else 0), self.n_envs, self.device
        outs = [torch.empty((N, 6, n), dtype=torch.float32, device=dev) if jac else None,
                torch.empty((N, n, n), dtype=torch.float32, device=dev) if mass else None,
                torch.empty((N, n), dtype=torch.float32, device=dev) if tau else None]
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        pt = (ctypes.c_float * 3)(*[float(x) for x in point])
        self._check(self.L.dg_body_dynamics(self._h, int(body), int(link), pt, p(q), p(qd), p(qdd), *[p(o) for o in outs], self._stream()))
        return tuple(outs)

    def body_ik(self, body, link, target_pos, target_orn=None, q=None, limits=None, max_iters=20, threshold=1e-4, err=False):
        """Inverse kinematics of body `body` for link `link` (dg_body_ik): new tensors (q [N, n_dof], err [N, 2] or None).
        target_pos [N, 3], target_orn [N, 4] or None, q [N, n_dof] or None (the state row's), limits [N, 4, n_dof] or None (no
        null-space term): contiguous float32 tensors on this world's device.  Asynchronous on the current stream."""
        nd, N, dev = self.scene.bodies[body].n_dofs, self.n_envs, self.device
        q_out = torch.empty((N, nd), dtype=torch.float32, device=dev)
        e = torch.empty((N, 2), dtype=torch.float32, device=dev) if err else None
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        self._check(self.L.dg_body_ik(self._h, int(body), int(link), p(target_pos), p(target_orn), p(q), p(limits), int(max_iters),
                                      float(threshold), p(q_out), p(e), self._stream()))
        return q_out, e

    # named views into the state / parameter rows (same names as csrc/scene_sections.h)
    def s(self, name, n):
        o = self.scene.hdr[name]
        return self.state[:, o:o + n]

    def p(self, name, n):
        o = self.scene.hdr[name]
        return self.param[:, o:o + n]
