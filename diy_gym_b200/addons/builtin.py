"""Built-in add-ons.  Each mirrors one class of `diy_gym/addons/**` in the reference: same config keys, same
spaces, same arithmetic - but the arithmetic is emitted as an op of the fused CUDA step (`compile`), and the
run-time hooks only move data in and out of the world's device buffers."""
import numpy as np
import torch

from .. import spaces
from .addon import Addon


def _is_model(parent):
    return hasattr(parent, 'body')


class _OpAddon(Addon):
    """Add-on backed by one scene op."""
    op = None

    def bind(self, env):
        self.env = env
        w, o = env.world, self.op
        if o is None:
            return
        self._act = w.action[:, o['act_off']:o['act_off'] + o['n_act']] if o['n_act'] else None
        self._obs = w.obs[:, o['obs_off']:o['obs_off'] + o['n_obs']] if o['n_obs'] else None
        self._rew = w.reward[:, o['rew_off']] if o['n_rew'] else None
        self._term = w.term[:, o['term_off']] if o['n_term'] else None

    def _put(self, dst, action):
        a = torch.as_tensor(action, device=dst.device, dtype=torch.float32)
        dst.copy_(a.reshape(-1, dst.shape[1]).expand_as(dst) if a.dim() else a.expand_as(dst))


class JointController(_OpAddon):
    """`controllers/joint_controller.py`: modes position / velocity (default) / torque on the named joints."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        b = parent.body
        self.mode = {'position': 0, 'velocity': 1, 'torque': 2}[config.get('control_mode', 'velocity')]
        names = b.joint_names()
        if 'joint' in config:
            joints = [config.get('joint')]
        elif 'joints' in config:
            joints = config.get('joints')
        else:
            joints = names
        # movable joints whose name was asked for, ordered by joint index (joint_controller.py:23-30)
        self.joint_ids = [i for i in range(b.num_joints()) if names[i] in joints and b.joint_dof[i] >= 0]
        n = len(self.joint_ids)
        self.rest_position = list(config.get('rest_position', [0] * n))
        self.torque_limit = [b.joint_info(i)['max_force'] for i in self.joint_ids]
        self.position_gain, self.velocity_gain = 0.03, 1.0   # joint_controller.py:53-58
        self.action_space = spaces.Box(-0.5, 0.5, shape=(n, ), dtype='float32')

    def compile(self, sb):
        b, n = self.parent.body, len(self.joint_ids)
        dofs = [b.global_dof(i) for i in self.joint_ids]
        self.op = sb.add_op('JOINT_CTRL', [self.mode, n] + dofs, [self.position_gain, self.velocity_gain] + self.torque_limit, n_act=n)
        m = min(n, len(self.rest_position))   # zip() truncation of joint_controller.py:36-38
        sb.add_op('JOINT_RESET', [m] + dofs[:m], self.rest_position[:m])

    def update(self, action):
        self._put(self._act, action)


class ExternalForce(_OpAddon):
    """`controllers/external_force.py`: force on the base at the world-space point `xyz` (WORLD_FRAME).
    Extension keys: `frame: link` applies force and point in the link frame, `link: <joint name>` picks a link."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.xyz = list(config.get('xyz', [0.0, 0.0, 0.0]))
        self.link = parent.get_frame_id(config.get('link')) if 'link' in config else -1
        self.link_frame = int(config.get('frame', 'world') == 'link')
        self.action_space = spaces.Box(-10.0, 10.0, shape=(3, ), dtype='float32')

    def compile(self, sb):
        self.op = sb.add_op('EXT_FORCE', [self.parent.body.frame(self.link), self.link_frame], self.xyz, n_act=3)

    def update(self, action):
        self._put(self._act, action)


class InverseKinematicsController(_OpAddon):
    resets_in_constructor = True   # ik_controller.py:45 calls self.reset(): a nested model is welded to the arm at its rest pose
    """`controllers/ik_controller.py`: end-effector pose delta -> damped-least-squares IK -> position motors."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        b = parent.body
        self.position_gain = config.get('position_gain', 0.015)
        self.velocity_gain = config.get('velocity_gain', 1.0)
        self.end_effector_joint_id = b.joint_names().index(config.get('end_effector'))
        self.joint_ids = [i for i in b.movable_joints() if i <= self.end_effector_joint_id]
        infos = [b.joint_info(i) for i in self.joint_ids]
        self.joint_position_lower_limit = [i['lower'] for i in infos]
        self.joint_position_upper_limit = [i['upper'] for i in infos]
        self.torque_limit = [i['max_force'] for i in infos]
        self.rest_position = list(config.get('rest_position', [0] * len(self.joint_ids)))
        self.use_orientation = bool(config.get('use_orientation', False))
        self.action_space = spaces.Dict({'linear': spaces.Box(-0.01, 0.01, shape=(3, ), dtype='float32')})
        if self.use_orientation:
            self.action_space.spaces['rotation'] = spaces.Box(-0.01, 0.01, shape=(3, ), dtype='float32')

    def compile(self, sb):
        b, n, ndb = self.parent.body, len(self.joint_ids), self.parent.body.n_dofs
        rest = self.rest_position
        # null-space terms only when the four lists span every DoF of the body (SURVEY App. A.4)
        nullspace = int(n == ndb and len(rest) == ndb)
        pad = lambda v: [float(x) for x in list(v)[:ndb]] + [0.0] * (ndb - min(len(v), ndb))
        rng = [u - l for l, u in zip(self.joint_position_lower_limit, self.joint_position_upper_limit)]
        fargs = [self.position_gain, self.velocity_gain] + self.torque_limit + pad(self.joint_position_lower_limit) + \
            pad(self.joint_position_upper_limit) + pad(rng) + pad(rest)
        dofs = [b.global_dof(i) for i in self.joint_ids]
        iargs = [b.index, b.link_start + self.end_effector_joint_id, n, int(self.use_orientation), nullspace] + dofs
        self.op = sb.add_op('IK_CTRL', iargs, fargs, n_act=6 if self.use_orientation else 3)
        m = min(n, len(rest))   # zip() truncation of ik_controller.py:47-49
        sb.add_op('JOINT_RESET', [m] + dofs[:m], rest[:m])

    def update(self, action):
        self._put(self._act[:, 0:3], action['linear'])
        if self.use_orientation:
            self._put(self._act[:, 3:6], action['rotation'])


class JointStateSensor(_OpAddon):
    """`sensors/joint_state_sensor.py`: position, velocity (default on), effort (default off)."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        b = parent.body
        if 'joints' in config:
            names = b.joint_names()
            self.joint_ids = [names.index(j) for j in config.get('joints')]
        else:
            self.joint_ids = b.movable_joints()
        self.include_velocity = bool(config.get('include_velocity', True))
        self.include_effort = bool(config.get('include_effort', False))
        infos = [b.joint_info(i) for i in self.joint_ids]
        lo, hi = np.array([i['lower'] for i in infos]), np.array([i['upper'] for i in infos])
        self.observation_space = spaces.Dict({'position': spaces.Box(low=lo, high=hi, dtype='float32')})
        if self.include_velocity:
            v = np.array([i['max_velocity'] for i in infos])
            self.observation_space.spaces['velocity'] = spaces.Box(low=-v, high=v, dtype='float32')
        if self.include_effort:
            t = np.array([i['max_force'] for i in infos])
            self.observation_space.spaces['effort'] = spaces.Box(low=-t, high=t, dtype='float32')

    def compile(self, sb):
        b, n = self.parent.body, len(self.joint_ids)
        if any(b.joint_dof[i] < 0 for i in self.joint_ids):
            raise ValueError('joint_state_sensor: fixed joints have no state')
        flags = int(self.include_velocity) | (int(self.include_effort) << 1)
        self.op = sb.add_op('JOINT_SENSOR', [n, flags] + [b.global_dof(i) for i in self.joint_ids],
                            n_obs=n * (1 + int(self.include_velocity) + int(self.include_effort)))

    def observe(self):
        n, o, j = len(self.joint_ids), self._obs, 1
        out = {'position': o[:, 0:n]}
        if self.include_velocity:
            out['velocity'] = o[:, j * n:(j + 1) * n]
            j += 1
        if self.include_effort:
            out['effort'] = o[:, j * n:(j + 1) * n]
        return out


class ObjectStateSensor(_OpAddon):
    """`sensors/object_state_sensor.py`: COM pose / twist of a model or frame, optionally relative to another."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.source_model = parent.models[config.get('source_model')] if 'source_model' in config else None
        self.target_model = parent.models[config.get('target_model')] if 'target_model' in config else parent
        self.source_frame_id = self.source_model.get_frame_id(config.get('source_frame')) if 'source_frame' in config else -1
        self.target_frame_id = self.target_model.get_frame_id(config.get('target_frame')) if 'target_frame' in config else -1
        self.include_rotation = bool(config.get('include_rotation', False))
        self.include_velocity = bool(config.get('include_velocity', False))
        box = lambda: spaces.Box(-10, 10, shape=(3, ), dtype='float32')
        self.observation_space = spaces.Dict({'position': box()})
        if self.include_rotation:
            self.observation_space.spaces['rotation'] = box()
        if self.include_velocity:
            self.observation_space.spaces['velocity'] = box()
        if self.include_rotation and self.include_velocity:
            self.observation_space.spaces['angular_velocity'] = box()

    def compile(self, sb):
        tf = self.target_model.body.frame(self.target_frame_id)
        sf = self.source_model.body.frame(self.source_frame_id) if self.source_model is not None else -1
        flags = int(self.include_rotation) | (int(self.include_velocity) << 1)
        n = 3 * (1 + int(self.include_rotation) + int(self.include_velocity) + int(self.include_rotation and self.include_velocity))
        self.op = sb.add_op('OBJECT_SENSOR', [tf, sf, flags], n_obs=n)

    def observe(self):
        o, j = self._obs, 3
        out = {'position': o[:, 0:3]}   # insertion order of object_state_sensor.py:64-73
        if self.include_velocity:
            out['velocity'] = o[:, j:j + 3]
            j += 3
        if self.include_rotation:
            out['rotation'] = o[:, j:j + 3]
            j += 3
        if self.include_rotation and self.include_velocity:
            out['angular_velocity'] = o[:, j:j + 3]
        return out


class Camera(Addon):
    """`sensors/camera.py`: rgb in [0,1] and eye-space depth from a camera on a frame of the parent (or fixed in
    the world for an environment-level camera), rendered by the batched ray-cast kernel on every observe()."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.near, self.far = config.get('clipping_boundaries', [0.01, 100])
        self.fov = config.get('field_of_view', 70.0)
        self.resolution = list(config.get('resolution', [640, 480]))
        self.frame_id = parent.get_frame_id(config.get('frame')) if 'frame' in config and _is_model(parent) else -1
        self.xyz = config.get('xyz', [0., 0., 0.])
        self.rpy = config.get('rpy', [0., 0., 0.])
        self.use_depth = bool(config.get('use_depth', True))
        self.use_seg_mask = bool(config.get('use_segmentation_mask', False))
        # extension key: the colour image as bytes (round(255 c), the renderer's own format - the reference divides it by 255,
        # camera.py:76-78): a quarter of the colour bytes for a host-side consumer to move
        self.rgb_uint8 = bool(config.get('rgb_uint8', False))
        self.observation_space = spaces.Dict({'rgb': spaces.Box(0, 255, shape=self.resolution + [3], dtype='uint8') if self.rgb_uint8
                                              else spaces.Box(0., 1., shape=self.resolution + [3], dtype='float32')})
        if self.use_depth:
            self.observation_space.spaces['depth'] = spaces.Box(0., 10., shape=self.resolution, dtype='float32')
        if self.use_seg_mask:   # camera.py:54-56
            self.observation_space.spaces['segmentation_mask'] = spaces.Box(0., 10., shape=self.resolution, dtype='float32')

    def compile(self, sb):
        from ..compiler.mathutil import quat_from_euler
        frame = self.parent.body.frame(self.frame_id) if _is_model(self.parent) else -1
        self.cam = sb.add_camera(frame, self.xyz, quat_from_euler(self.rpy), self.resolution[0], self.resolution[1], self.fov, self.near, self.far)

    def bind(self, env):
        self.env = env

    def observe(self):
        img = self.env.world.render(self.cam, seg=self.use_seg_mask, u8=self.rgb_uint8)
        out = {'rgb': img[0]}   # [N, H, W, 3]; the reference labels the same buffer (W, H, 3) (camera.py:77)
        if self.use_depth:
            out['depth'] = img[1]
        if self.use_seg_mask:   # unique id of the visible body per pixel, -1 = background (camera.py:89-90)
            out['segmentation_mask'] = img[2]
        return out


class ReachTarget(_OpAddon):
    """`rewards/reach_target.py`: -distance * multiplier between two frames, terminal below `tolerance`."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.source_model = parent.models[config.get('source_model')]
        self.target_model = parent.models[config.get('target_model')]
        self.source_frame_id = self.source_model.get_frame_id(config.get('source_frame')) if 'source_frame' in config else -1
        self.target_frame_id = self.target_model.get_frame_id(config.get('target_frame')) if 'target_frame' in config else -1
        self.multiplier = config.get('multiplier', 1.0)
        self.tolerance = config.get('tolerance', 0.05)

    def compile(self, sb):
        self.op = sb.add_op('REACH_TARGET', [self.source_model.body.frame(self.source_frame_id), self.target_model.body.frame(self.target_frame_id)],
                            [self.multiplier, self.tolerance], n_rew=1, n_term=1)

    def reward(self):
        return self._rew

    def is_terminal(self):
        return self._term.bool()


class ElectricityCost(_OpAddon):
    """`rewards/electricity_cost.py`: -sum |motor torque * joint velocity| * multiplier over all movable joints."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.multiplier = config.get('multiplier', 1.0)

    def compile(self, sb):
        self.op = sb.add_op('ELECTRICITY', [self.parent.body.index], [self.multiplier], n_rew=1)

    def reward(self):
        return self._rew


class StuckJointCost(_OpAddon):
    """`rewards/stuck_joint_cost.py` (the reference raises NameError; this implements its stated intent:
    -multiplier when any joint is within 0.01 of a limit)."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.multiplier = config.get('multiplier', 0.1)

    def compile(self, sb):
        self.op = sb.add_op('STUCK_JOINT', [self.parent.body.index], [self.multiplier], n_rew=1)

    def reward(self):
        return self._rew


class TimePenalty(_OpAddon):
    """`rewards/time_penalty.py`: constant `penalty` per step (default -1)."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.penalty = config.get('penalty', -1)

    def compile(self, sb):
        self.op = sb.add_op('TIME_PENALTY', [], [self.penalty], n_rew=1)

    def reward(self):
        return self._rew


class Respawn(_OpAddon):
    """`misc/respawn.py`: on reset, base pose = initial pose jittered uniformly within position / rotation range.
    Random numbers come from the per-environment counter-based stream (seed, env id, reset count)."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.position_range = list(config.get('position_range', [0., 0., 0.]))
        self.rotation_range = list(config.get('rotation_range', [0., 0., 0.]))
        self.once = bool(config.get('once', False))
        parent.body.per_env_pose = True

    def compile(self, sb):
        self.op = sb.add_op('RESPAWN', [self.parent.body.index, int(self.once)], self.position_range + self.rotation_range)


class DynamicsRandomizer(_OpAddon):
    """`misc/dynamics_randomizer.py`: per reset, link masses and joint damping scaled log-uniformly within the
    ranges - applied to the NOMINAL values (the reference multiplies by log(U) and compounds; SURVEY App. D.6)."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.mass_range = list(config.get('mass_range', [0.25, 4.0]))
        self.damping_range = list(config.get('damping_range', [0.2, 20]))
        # extension keys (BASELINE.json config 5 / SURVEY 8d): lateral friction drawn uniformly per environment and reset, and a
        # nominal joint damping for models whose URDF gives none (the UR5: damping 0, so damping_range alone would do nothing)
        self.friction_range = [float(v) for v in config.get('friction_range', [0.0, 0.0])]
        self.nominal_damping = float(config.get('nominal_damping', 0.0))

    def compile(self, sb):
        self.op = sb.add_op('DYN_RANDOMIZE', [self.parent.body.index], self.mass_range + self.damping_range + self.friction_range + [self.nominal_damping])


class SpawnMultiple(Addon):
    """`misc/spawn_multiple.py`: clone the nested model `num_models` times into the parent's models."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        from ..model import Model
        child = config.find('model')
        for i in range(config.get('num_models')):
            cfg = type(child)(child.name + '_%d' % i, child.node)
            parent.models[cfg.name] = Model(cfg, env=parent if not _is_model(parent) else parent.env)


class DrawCoords(Addon):
    """`misc/draw_coords.py` draws GUI debug lines; headless batched simulation has no GUI, so this is a no-op."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.action_space = spaces.Box(-1., 1., shape=(0, ), dtype='float32')


class _Unsupported(Addon):
    reason = ''

    def __init__(self, parent, config):
        raise NotImplementedError('%s: %s' % (config.get('addon'), self.reason))


class AdmittanceController(_OpAddon):
    resets_in_constructor = True   # admittance_controller.py:34
    """`controllers/admittance_controller.py`: joint torques = F . J_lin + T . J_ang (Jacobian of the admittance point on the
    end effector) + gravity compensation + p_gain (target_pose - q) - d_gain qd; the default joint motors are switched off."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        b = parent.body
        self.end_frame = parent.get_frame_id(config.get('end_effector'))
        self.offset_admittance_point = list(config.get('offset_admittance_point', [0., 0., 0.]))
        self.kp = config.get('p_gain', 0.001)
        self.kd = config.get('d_gain', 0.01)
        self.joint_ids = [i for i in b.movable_joints() if i <= self.end_frame]
        n = len(self.joint_ids)
        # p.calculateInverseDynamics(uid, joint_positions, ...) (admittance_controller.py:47) takes one position per DoF of
        # the body: a joint list that leaves DoF out makes pybullet raise, and so does a floating base
        if n != b.n_dofs or b.kind != 1:
            raise ValueError('admittance_controller: the joints up to end_effector must span every DoF of a fixed-base model '
                             '(%d of %d)' % (n, b.n_dofs))
        self.rest_position = list(config.get('rest_position', [0] * n))
        self.target_pose = list(config.get('target_pose', self.rest_position))
        if len(self.target_pose) != n:
            raise ValueError('admittance_controller: target_pose needs %d entries' % n)
        self.action_space = spaces.Dict({'force': spaces.Box(-5, 5, shape=(3, ), dtype='float32'),
                                         'torque': spaces.Box(-1., 1., shape=(3, ), dtype='float32')})

    def compile(self, sb):
        b, n = self.parent.body, len(self.joint_ids)
        dofs = [b.global_dof(i) for i in self.joint_ids]
        self.op = sb.add_op('ADMITTANCE', [b.index, b.link_start + self.end_frame, n] + dofs,
                            [self.kp, self.kd] + self.offset_admittance_point + self.target_pose, n_act=6)
        m = min(n, len(self.rest_position))   # zip() truncation of admittance_controller.py:36-38
        sb.add_op('JOINT_RESET', [m] + dofs[:m], self.rest_position[:m])
        sb.motors_off += dofs                  # VELOCITY_CONTROL with forces = 0 (admittance_controller.py:34)

    def update(self, action):
        self._put(self._act[:, 0:3], action['force'])
        self._put(self._act[:, 3:6], action['torque'])


class ForceTorqueSensor(_OpAddon):
    """`sensors/force_torque_sensor.py`: joint reaction force / torque of the joint `frame` (p.getJointState(...)[2] after
    enableJointForceTorqueSensor), expressed in the child link's COM frame, from the forward-dynamics pass of the last sub-step."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.frame_id = parent.get_frame_id(config.get('frame')) if 'frame' in config else -1
        if self.frame_id < 0:   # p.getJointState(uid, -1) raises in the reference as well (force_torque_sensor.py:22)
            raise ValueError('force_torque_sensor: `frame` must name a joint of the model')
        box = lambda: spaces.Box(-10, 10, shape=(3, ), dtype='float32')
        self.observation_space = spaces.Dict({'force': box(), 'torque': box()})

    def compile(self, sb):
        sb.need_jreact = True
        self.op = sb.add_op('FT_SENSOR', [self.parent.body.link_start + self.frame_id], n_obs=6)

    def observe(self):
        return {'force': self._obs[:, 0:3], 'torque': self._obs[:, 3:6]}


class VisualRandomizer(_OpAddon):
    """`misc/visual_randomizer.py`: a new look for the parent model on every reset.  The reference applies a random texture of a
    dataset it downloads on first use (visual_randomizer.py:41-60); this backend has no textures, so the randomisation is a random
    colour per visual shape of the model, per environment and reset, from the same counter-based stream as respawn /
    dynamics_randomizer (op `VIS_RANDOMIZE`, stored in the parameter rows, read by the camera kernel)."""
    def compile(self, sb):
        self.op = sb.add_op('VIS_RANDOMIZE', [self.parent.body.index], [])


class FilteredLinkWrench(_OpAddon):
    """Building block for USER add-ons that would otherwise run as eager PyTorch every step: a scalar action in [0, 1] goes
    through a first-order filter (state += (action - state) * rate) and scales a force and a torque given in the frame of a
    link (applyExternalForce / applyExternalTorque with LINK_FRAME).  One op of the fused step (`FILTERED_WRENCH`); the filter
    state lives in the state row and is the add-on's observation.  The reference's examples/drone_pilot `Propellor`
    (drone_pilot.py:10-40) is exactly this - examples/drone_pilot/drone_pilot.py subclasses it.
    Keys: frame (joint name, default base), force [3], torque [3], position [3] (point of application, link frame), rate,
    reset_state (default no: the reference's Propellor keeps its rotor speed across resets)."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.frame_id = parent.get_frame_id(config.get('frame')) if 'frame' in config else -1
        self.force = [float(v) for v in config.get('force', [0.0, 0.0, 0.0])]
        self.torque = [float(v) for v in config.get('torque', [0.0, 0.0, 0.0])]
        self.position = [float(v) for v in config.get('position', [0.0, 0.0, 0.0])]
        self.rate = float(config.get('rate', 0.1))
        self.reset_state = bool(config.get('reset_state', False))
        self.observation_space = spaces.Box(0.0, 1.0, shape=(1, ), dtype='float32')
        self.action_space = spaces.Box(0.0, 1.0, shape=(1, ), dtype='float32')

    def compile(self, sb):
        slot = sb.alloc_addon_state(1)
        self.op = sb.add_op('FILTERED_WRENCH', [self.parent.body.frame(self.frame_id), int(self.reset_state), slot],
                            [self.rate] + self.force + self.torque + self.position, n_act=1, n_obs=1)

    def update(self, action):
        self._put(self._act, action)

    def observe(self):
        return self._obs


class TiltTerminal(_OpAddon):
    """Terminal when the base of the parent model is tilted by more than `angle` degrees (op `TILT_TERMINAL`); the reference's
    examples/drone_pilot `FellOver` (drone_pilot.py:43-55) with its 10 degrees."""
    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.angle = float(config.get('angle', 10.0))

    def compile(self, sb):
        self.op = sb.add_op('TILT_TERMINAL', [self.parent.body.index], [float(np.radians(self.angle))], n_term=1)

    def is_terminal(self):
        return self._term.bool()


class RaySensor(_OpAddon):
    """Range finder (pybullet's rayTestBatch): rays from a point on a frame of the parent (or fixed in the world for an
    environment-level sensor) against the collision shapes of every body, the parent included.  Per ray the distance to the first
    surface the ray enters with t in (min, max] (max on a miss) and, with `include_hit_object`, the body index hit (load order, as
    pybullet's uid and the segmentation mask; -1 on a miss).  Cast by dg_ray_kernel after every step / reset / observe (op
    `RAY_SENSOR`).  Keys: frame (joint name, default the base), xyz, rpy (sensor pose in that frame, the camera's convention), range
    [min, max], num_rays / horizontal_fov / vertical_angles (a pattern about the sensor's z axis: azimuths k 360 / n over a full
    turn, else -fov/2 .. +fov/2 inclusive; one layer per elevation in degrees, layer-major) or `directions` (explicit, in the
    sensor frame, normalised), include_hit_object."""
    MAX_RAYS = 1024

    def __init__(self, parent, config):
        super().__init__(parent, config)
        self.frame_id = -1
        if 'frame' in config:
            names = parent.body.joint_names() if _is_model(parent) else []
            if config.get('frame') not in names:
                raise ValueError('ray_sensor: unknown frame %r' % (config.get('frame'), ))
            self.frame_id = parent.get_frame_id(config.get('frame'))
        self.xyz = [float(v) for v in config.get('xyz', [0.0, 0.0, 0.0])]
        self.rpy = [float(v) for v in config.get('rpy', [0.0, 0.0, 0.0])]
        rng = [float(v) for v in config.get('range', [0.0, 10.0])]
        if len(rng) != 2:
            raise ValueError('ray_sensor: range must be [min, max]')
        self.min, self.max = rng
        if self.min < 0 or self.min >= self.max:
            raise ValueError('ray_sensor: range needs 0 <= min < max (got %r)' % (rng, ))
        self.include_hit_object = bool(config.get('include_hit_object', False))
        if 'directions' in config:
            d = np.asarray(config.get('directions'), float).reshape(-1, 3)
            n = np.linalg.norm(d, axis=1)
            if d.shape[0] < 1 or np.any(n == 0):
                raise ValueError('ray_sensor: directions must be non-empty and of non-zero length')
            self.directions = d / n[:, None]
        else:
            self.directions = self.pattern(int(config.get('num_rays', 1)), float(config.get('horizontal_fov', 360.0)),
                                           [float(v) for v in config.get('vertical_angles', [0.0])])
        self.num_rays = len(self.directions)
        if self.num_rays > self.MAX_RAYS:
            raise ValueError('ray_sensor: %d rays, at most %d per sensor' % (self.num_rays, self.MAX_RAYS))
        self.observation_space = spaces.Dict({'distance': spaces.Box(self.min, self.max, shape=(self.num_rays, ), dtype='float32')})
        if self.include_hit_object:
            self.observation_space.spaces['hit_object'] = spaces.Box(-1.0, np.inf, shape=(self.num_rays, ), dtype='float32')

    @staticmethod
    def pattern(num_rays, horizontal_fov, vertical_angles):
        """Unit directions of the pattern, layer-major: azimuths about z, one layer per elevation (degrees)."""
        if num_rays < 1:
            raise ValueError('ray_sensor: num_rays must be at least 1')
        if not 0.0 < horizontal_fov <= 360.0:
            raise ValueError('ray_sensor: horizontal_fov must be in (0, 360]')
        if len(vertical_angles) < 1:
            raise ValueError('ray_sensor: vertical_angles needs at least one elevation')
        k = np.arange(num_rays, dtype=float)
        if horizontal_fov == 360.0:
            az = k * 360.0 / num_rays
        else:
            az = -horizontal_fov / 2 + k * (horizontal_fov / (num_rays - 1)) if num_rays > 1 else np.zeros(1)
        az = np.radians(az)
        out = []
        for el in np.radians(np.asarray(vertical_angles, float)):
            out.append(np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.full_like(az, np.sin(el))], axis=1))
        return np.concatenate(out, axis=0)

    def compile(self, sb):
        from ..compiler.mathutil import quat_from_euler
        frame = self.parent.body.frame(self.frame_id) if _is_model(self.parent) else -1
        R = self.num_rays
        self.op = sb.add_op('RAY_SENSOR', [frame, R, int(self.include_hit_object)],
                            self.xyz + list(quat_from_euler(self.rpy)) + [self.min, self.max] + self.directions.reshape(-1).tolist(),
                            n_obs=2 * R if self.include_hit_object else R)

    def observe(self):
        R = self.num_rays
        out = {'distance': self._obs[:, 0:R]}
        if self.include_hit_object:
            out['hit_object'] = self._obs[:, R:2 * R]
        return out


BUILTIN_ADDONS = {
    'ray_sensor': RaySensor,
    'filtered_link_wrench': FilteredLinkWrench, 'tilt_terminal': TiltTerminal,
    'ik_controller': InverseKinematicsController, 'joint_controller': JointController, 'admittance_controller': AdmittanceController,
    'camera': Camera, 'joint_state_sensor': JointStateSensor, 'object_state_sensor': ObjectStateSensor,
    'force_torque_sensor': ForceTorqueSensor, 'reach_target': ReachTarget, 'stuck_joint_cost': StuckJointCost,
    'electricity_cost': ElectricityCost, 'time_penalty': TimePenalty, 'respawn': Respawn, 'spawn_multiple': SpawnMultiple,
    'draw_coords': DrawCoords, 'external_force': ExternalForce, 'visual_randomizer': VisualRandomizer,
    'dynamics_randomizer': DynamicsRandomizer,
}
