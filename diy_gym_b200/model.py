"""Model: one spawned URDF (what `diy_gym/model.py:11-106` of the reference builds through pybullet).

At construction a Model registers its body with the scene builder (north_star (a): URDF -> SoA buffers) and
creates its add-ons and nested models; at run time it is a thin view on the batched device state for user
add-ons: every query returns torch tensors with leading dimension `num_envs`.

Config keys, as in the reference (`model.py:34-47`): model, xyz, rpy, scale, use_fixed_base, mass, color,
parent_frame, child_frame.
"""
from collections import OrderedDict

import numpy as np
import torch

from . import torch_math as tm
from .addons.addon import AddonFactory, Receptor
from .assets import resolve_model
from .backend import DYN_MAX_N, IK_MAX_ND
from .compiler.mathutil import quat_from_euler


class Model(Receptor):
    def __init__(self, config, parent=None, env=None):
        Receptor.__init__(self)
        self.name = config.name
        self.env = env if env is not None else parent.env
        self.position = config.get('xyz', [0., 0., 0.])
        self.orientation = quat_from_euler(config.get('rpy', [0., 0., 0.]))
        use_fixed_base = config.get('use_fixed_base', False)
        scale = config.get('scale', 1.0)
        urdf = config.get('model')
        desc = resolve_model(urdf)   # raises ValueError('Could not find URDF: ...') like model.py:63
        spawn_pos, spawn_quat = self.position, self.orientation
        if parent is not None:
            # model.py:69-77: the child is spawned at the COM pose of the parent frame (getLinkState[:2] / base pose) and welded
            # to it with p.createConstraint(JOINT_FIXED): joint frame = (xyz, rpy) in the parent frame, identity in the child frame
            parent_frame_id = parent.get_frame_id(config.get('parent_frame')) if 'parent_frame' in config else -1
            # (the parent's controllers have already put its joints at their rest_position: add-ons are built before nested models)
            # - but only the controllers whose constructor calls reset() in the reference do that (ik_controller.py:45,
            # admittance_controller.py:34); under a joint_controller the parent is still at q = 0 when the child is welded
            q_rest = {}
            for a in parent.addons.values():
                if getattr(a, 'resets_in_constructor', False) and hasattr(a, 'joint_ids') and hasattr(a, 'rest_position'):
                    q_rest.update(dict(zip(a.joint_ids, a.rest_position)))
            T = parent.body.rest_com_pose(parent_frame_id, q_rest)
            spawn_pos, spawn_quat = T.p, T.q
        self.body = self.env.builder.add_body(self.name, desc, xyz=spawn_pos, quat=spawn_quat, scale=scale,
                                              fixed_base=use_fixed_base, mass=config.get('mass') if 'mass' in config else None,
                                              color=config.get('color') if 'color' in config else None)
        if parent is not None:
            child_frame_id = self.get_frame_id(config.get('child_frame')) if 'child_frame' in config else -1
            self.env.builder.add_fixed_constraint(parent.body, parent_frame_id, self.body, child_frame_id, self.position, self.orientation)
        self.uid = self.body.index
        self.addons = OrderedDict(sorted({child.name: AddonFactory.build(child.get('addon'), self, child)
                                          for child in config.find_all('addon')}.items(), key=lambda t: t[0]))
        self.models = OrderedDict(sorted({child.name: Model(child, self) for child in config.find_all('model')}.items(),
                                         key=lambda t: t[0]))

    # ---- pybullet-like introspection (compile time) -----------------------------------------------
    def get_frame_id(self, frame):
        """Joint index of the named joint / frame, -1 for the base or an unknown name (`model.py:94-96`)."""
        return self.body.joint_index(frame)

    def num_joints(self):
        return self.body.num_joints()

    def joint_info(self, i):
        return self.body.joint_info(i)

    # ---- batched state views (run time) --------------------------------------------------------
    @property
    def world(self):
        return self.env.world

    def _h(self, name):
        return self.env.scene.hdr[name]

    def base_pose(self):
        """COM pose of the base: ([N,3], [N,4] xyzw) - getBasePositionAndOrientation."""
        b, st = self.uid, self.world.state
        return st[:, self._h('S_BPOS') + 3 * b:self._h('S_BPOS') + 3 * b + 3], st[:, self._h('S_BQUAT') + 4 * b:self._h('S_BQUAT') + 4 * b + 4]

    def base_velocity(self):
        b, st = self.uid, self.world.state
        return st[:, self._h('S_BVEL') + 3 * b:self._h('S_BVEL') + 3 * b + 3], st[:, self._h('S_BOMEGA') + 3 * b:self._h('S_BOMEGA') + 3 * b + 3]

    def link_state(self, frame_id):
        """COM-frame pose and world velocity of link `frame_id` (-1 = base) as cached after the last step:
        (pos, quat, lin_vel, ang_vel) - getLinkState[0,1,6,7] with computeLinkVelocity=1."""
        if frame_id < 0:
            return self.base_pose() + self.base_velocity()
        gl, st = self.body.link_start + frame_id, self.world.state
        return (st[:, self._h('S_LPOS') + 3 * gl:self._h('S_LPOS') + 3 * gl + 3], st[:, self._h('S_LQUAT') + 4 * gl:self._h('S_LQUAT') + 4 * gl + 4],
                st[:, self._h('S_LVEL') + 3 * gl:self._h('S_LVEL') + 3 * gl + 3], st[:, self._h('S_LOMEGA') + 3 * gl:self._h('S_LOMEGA') + 3 * gl + 3])

    def get_transform(self, frame_id=-1):
        """URDF link-frame pose (getLinkState[4,5]) or the base pose (`model.py:98-106`)."""
        if frame_id < 0:
            return self.base_pose()
        pos, quat, _, _ = self.link_state(frame_id)
        lf = self.env.scene.sec['LINK_F'][self.body.link_start + frame_id]
        d = pos.new_tensor(lf[7:10])
        qi = quat.new_tensor([-lf[16], -lf[17], -lf[18], lf[19]])
        return pos - tm.quat_rotate(quat, d.expand_as(pos)), tm.quat_mul(quat, qi.expand_as(quat))

    def joint_state(self, joint_ids=None):
        """(q, qd, applied motor torque) for the given joint indices (default: all movable) - getJointStates[0,1,3]."""
        ids = self.body.movable_joints() if joint_ids is None else list(joint_ids)
        dofs = [self.body.global_dof(i) for i in ids]
        st, dt = self.world.state, self.env.scene.hdr_f['dt']
        idx = torch.as_tensor(dofs, device=st.device, dtype=torch.long)
        return st[:, self._h('S_Q') + idx], st[:, self._h('S_QD') + idx], st[:, self._h('S_MAPPLIED') + idx] / dt

    def _frame(self, link):
        return self.body.frame(link)

    def apply_external_force(self, link, force, position=None, frame='world'):
        """Batched applyExternalForce: force [N,3] (or [3]) on link (-1 = base) at `position`, both given in
        the WORLD frame or in the LINK (COM) frame; acts during the next step only."""
        st = self.world.state
        f = self._frame(link)
        force = torch.as_tensor(force, device=st.device, dtype=torch.float32).expand(st.shape[0], 3)
        pos, quat, _, _ = self.link_state(link)
        if position is None:
            position = pos if frame == 'world' else torch.zeros_like(pos)
        position = torch.as_tensor(position, device=st.device, dtype=torch.float32).expand(st.shape[0], 3)
        if frame == 'link':
            force = tm.quat_rotate(quat, force)
            rel = tm.quat_rotate(quat, position)
        else:
            rel = position - pos
        o_f, o_t = self._h('S_EXTF') + 3 * f, self._h('S_EXTT') + 3 * f
        st[:, o_f:o_f + 3] += force
        st[:, o_t:o_t + 3] += torch.cross(rel, force, dim=-1)

    def apply_external_torque(self, link, torque, frame='world'):
        st = self.world.state
        f = self._frame(link)
        torque = torch.as_tensor(torque, device=st.device, dtype=torch.float32).expand(st.shape[0], 3)
        if frame == 'link':
            torque = tm.quat_rotate(self.link_state(link)[1], torque)
        o_t = self._h('S_EXTT') + 3 * f
        st[:, o_t:o_t + 3] += torque

    def apply_joint_torque(self, joint_ids, torque):
        """Batched setJointMotorControlArray(TORQUE_CONTROL): adds torque [N, len(joint_ids)] (or anything that broadcasts to it)
        to the applied joint torque of those movable joints; acts during the next step only, like apply_external_force."""
        cols = self._dofs(joint_ids, 'apply_joint_torque')
        st = self.world.state
        try:
            torque = torch.as_tensor(torque, device=st.device, dtype=torch.float32).expand(st.shape[0], len(cols))
        except RuntimeError as e:
            raise ValueError('apply_joint_torque: torque must broadcast to [%d, %d] (%s)' % (st.shape[0], len(cols), e))
        st.index_add_(1, torch.as_tensor(cols, device=st.device) + self._h('S_JTORQUE'), torque)

    def disable_motors(self, joint_ids):
        """setJointMotorControlArray(VELOCITY_CONTROL, forces=0): switches off the default velocity motor of those movable joints
        in every environment (the scene's default state).  Constructor-time only: call it from an add-on's __init__."""
        dofs = self._dofs(joint_ids, 'disable_motors')
        if self.env.builder.finalized is not None:
            raise ValueError('disable_motors: the scene is already compiled; call it from an add-on constructor')
        self.env.builder.motors_off += dofs

    def _dofs(self, joint_ids, what):
        ids, movable = list(joint_ids), set(self.body.movable_joints())
        bad = [i for i in ids if i not in movable]
        if bad:
            raise ValueError('%s: joints %s of %s are not movable joints (fixed or unknown)' % (what, bad, self.name))
        return [self.body.global_dof(i) for i in ids]

    # ---- rigid-body dynamics queries (dg_body_dynamics) ----------------------------------------------
    # Generalized velocity nu: [omega_base (world), v_base (world, base COM), qd] for a floating base, qd for a fixed one, with qd
    # in movable_joints() order; n = len(nu).  q [N, n_dof] holds joint positions only: the base pose is the state row's.
    def jacobian(self, frame_id=-1, local_position=(0., 0., 0.), q=None):
        """calculateJacobian: (J_lin [N, 3, n], J_ang [N, 3, n]) in world axes of the point `local_position`, given in the COM frame
        of link `frame_id` (-1 = base), at joint positions q (None: the state's)."""
        if not -1 <= int(frame_id) < self.num_joints():
            raise ValueError('jacobian: frame %d out of range [-1, %d)' % (frame_id, self.num_joints()))
        p = [float(x) for x in np.asarray(local_position, float).reshape(-1)]
        if len(p) != 3:
            raise ValueError('jacobian: local_position needs 3 entries')
        J = self._dynamics(int(frame_id), p, q, None, None, jac=True)[0]
        return J[:, :3], J[:, 3:]

    def mass_matrix(self, q=None):
        """calculateMassMatrix: M [N, n, n] at joint positions q (None: the state's); masses and inertias of the parameter row."""
        return self._dynamics(-1, (0., 0., 0.), q, None, None, mass=True)[1]

    def inverse_dynamics(self, q=None, qd=None, qdd=None):
        """calculateInverseDynamics: tau [N, n] = M(q) qdd + C(q, nu) nu + G(q) with the scene's gravity (None: the state's q, the
        state's nu, zero qdd).  For a floating base tau[:, :6] is the base wrench [torque about the base COM, force], world axes.
        Joint damping, motors, limits and contacts are not included."""
        return self._dynamics(-1, (0., 0., 0.), q, qd, qdd, tau=True)[2]

    def _dynamics(self, link, point, q, qd, qdd, jac=False, mass=False, tau=False):
        n = self.body.n_dofs + (6 if self.body.kind == 2 else 0)
        if n == 0:
            raise ValueError('%s has no degrees of freedom: no dynamics to query' % self.name)
        if n > DYN_MAX_N:
            raise ValueError('%s has %d generalized coordinates; the dynamics queries take at most %d' % (self.name, n, DYN_MAX_N))
        st = self.world.state
        args = []
        for name, t, width in (('q', q, self.body.n_dofs), ('qd', qd, n), ('qdd', qdd, n)):
            if t is not None:
                if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or t.device != st.device or tuple(t.shape) != (st.shape[0], width):
                    raise ValueError('%s must be a float32 tensor of shape [%d, %d] on %s' % (name, st.shape[0], width, st.device))
                t = t.contiguous()
            args.append(t)
        return self.world.body_dynamics(self.uid, link, point, *args, jac=jac, mass=mass, tau=tau)

    # ---- inverse kinematics (dg_body_ik) and position motors -------------------------------------------
    def inverse_kinematics(self, frame_id, target_position, target_orientation=None, q=None, lower_limits=None, upper_limits=None,
                           joint_ranges=None, rest_poses=None, max_iterations=None, residual_threshold=None, return_error=False):
        """calculateInverseKinematics for every environment: q [N, n_dof] (movable_joints() order) that brings the URDF frame of
        link `frame_id` to target_position ([N, 3] or [3], world) and, if given, target_orientation ([N, 4] or [4], xyzw, world;
        None: position only).  The ik_controller op's damped least squares, in the coordinates of the base, whose pose is the
        state's and stays fixed: from the seed q ([N, n_dof]; None: the state's q), at most max_iterations iterations (None: the
        scene's ik_iters) while the position residual exceeds residual_threshold (None: the scene's ik_threshold).
        lower_limits, upper_limits, joint_ranges, rest_poses ([n_dof] or [N, n_dof]): all four add the null-space term; giving
        only some, or lists of another length, raises ValueError (pybullet silently solves without the term then).
        return_error=True returns (q, err): err [N, 2] is the link frame's distance from the target (m) and the angle of the
        remaining rotation (rad, 0 without an orientation) at the returned q.  Inputs are float32 tensors on the world's device;
        nothing waits for the GPU."""
        if not 0 <= int(frame_id) < self.num_joints():
            raise ValueError('inverse_kinematics: frame %d out of range [0, %d): the target must be a link' % (frame_id, self.num_joints()))
        nd = self.body.n_dofs
        if nd == 0:
            raise ValueError('%s has no degrees of freedom: nothing to solve for' % self.name)
        if nd > IK_MAX_ND:
            raise ValueError('%s has %d degrees of freedom; inverse_kinematics takes at most %d' % (self.name, nd, IK_MAX_ND))
        sc = self.env.scene
        iters = sc.hdr['ik_iters'] if max_iterations is None else max_iterations
        thr = sc.hdr_f['ik_threshold'] if residual_threshold is None else residual_threshold
        if int(iters) != iters or iters < 1:
            raise ValueError('inverse_kinematics: max_iterations must be an integer >= 1, got %r' % (iters, ))
        if not float(thr) >= 0:
            raise ValueError('inverse_kinematics: residual_threshold must be >= 0, got %r' % (thr, ))
        tpos = self._batched('target_position', target_position, 3)
        torn = None if target_orientation is None else self._batched('target_orientation', target_orientation, 4)
        if q is not None:
            q = self._batched('q', q, nd, single=False)
        lists = (('lower_limits', lower_limits), ('upper_limits', upper_limits), ('joint_ranges', joint_ranges), ('rest_poses', rest_poses))
        given = [v is not None for _, v in lists]
        lim = None
        if any(given):
            if not all(given):
                raise ValueError('inverse_kinematics: give all of lower_limits, upper_limits, joint_ranges and rest_poses, or none')
            lim = torch.stack([self._batched(name, v, nd) for name, v in lists], 1).contiguous()
        q_out, err = self.world.body_ik(self.uid, int(frame_id), tpos, torn, q, lim, int(iters), float(thr), bool(return_error))
        return (q_out, err) if return_error else q_out

    def _batched(self, name, t, width, single=True):
        """t as a contiguous [N, width] tensor: a float32 tensor on the world's device of shape [N, width] (or [width] if single)."""
        st = self.world.state
        N = st.shape[0]
        shapes = [(N, width)] + ([(width, )] if single else [])
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or t.device != st.device or tuple(t.shape) not in shapes:
            raise ValueError('%s must be a float32 tensor of shape %s on %s' % (name, ' or '.join(str(list(s)) for s in shapes), st.device))
        return t.expand(N, width).contiguous()

    def set_position_targets(self, joint_ids, target, position_gain=0.03, velocity_gain=1.0, max_force=None):
        """setJointMotorControlArray(POSITION_CONTROL): the motors of those movable joints drive them to target with the gains
        position_gain (on the position error) and velocity_gain (on the velocity error, target velocity 0), with at most max_force
        (None: the URDF effort of each joint, as joint_controller).  Each value is a scalar or broadcasts to
        [N, len(joint_ids)].  These are the motor fields the joint_controller op writes in position mode.  Like pybullet's motor
        settings they persist until changed: reset() does not restore them, and a built-in controller op on the same joints
        overwrites them during the step (ops run inside the kernel, after update())."""
        ids = list(joint_ids)
        st = self.world.state
        cols = torch.as_tensor(self._dofs(ids, 'set_position_targets'), device=st.device)
        if max_force is None:
            max_force = [self.body.joint_info(i)['max_force'] for i in ids]
        vals = []
        for name, field, v in (('target', 'S_MTPOS', target), ('position_gain', 'S_MKP', position_gain),
                               ('velocity_gain', 'S_MKD', velocity_gain), ('max_force', 'S_MMAXF', max_force)):
            try:
                vals.append((field, torch.as_tensor(v, device=st.device, dtype=torch.float32).expand(st.shape[0], len(ids))))
            except RuntimeError as e:
                raise ValueError('set_position_targets: %s must broadcast to [%d, %d] (%s)' % (name, st.shape[0], len(ids), e))
        for field, v in vals:
            st[:, cols + self._h(field)] = v
        st[:, cols + self._h('S_MTVEL')] = 0.0
