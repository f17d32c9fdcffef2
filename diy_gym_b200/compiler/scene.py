"""Scene compiler: model descriptors + spawn poses + add-on programs -> flat SoA description.

This is north_star (a): "URDF/config compilation into SoA device buffers of links, joints, inertias and
primitive collision shapes, with per-env randomised parameters".  It replaces everything the reference
does at construction time through `p.loadURDF / resetBasePositionAndOrientation / changeDynamics`
(`diy_gym/model.py:48-92`) and through add-on constructors querying `p.getJointInfo`.

The result is two flat buffers (`ibuf` int32, `fbuf` float64) with a section table
(see `SECTIONS`); the CPU oracle and the CUDA backend each parse them independently.

Multibody convention (own restatement; equivalent to the reference engine's, SURVEY.md App. A.1):
every link frame used by the dynamics is the link's inertial (COM) frame.  For link i with parent P:
    T_Pcom_icom(q) = [ R0 * Rot(a, q),  e + R(q) d ]            (revolute)
                     [ R0,              e + R0 (d + a q) ]      (prismatic)
with  R0/e from  LP^-1 * parent2joint,  d = LI.R^T LI.p,  a = LI.R^T axis  (LP/LI = local inertial frames).
"""
from collections import OrderedDict

import numpy as np

from .mathutil import Transform, quat_from_euler, quat_to_mat, quat_mul, quat_conj, quat_rotate
from .urdf import inertia_from_rule

# ---- section ids (order is the ABI between Python and both C parsers) -------------------------------
SECTIONS = [
    ('HDR_I', 'i'), ('HDR_F', 'f'), ('BODY_I', 'i'), ('BODY_F', 'f'), ('LINK_I', 'i'), ('LINK_F', 'f'), ('SHAPE_I', 'i'),
    ('SHAPE_F', 'f'), ('PAIR_I', 'i'), ('VIS_I', 'i'), ('VIS_F', 'f'), ('OP_I', 'i'), ('OPARG_I', 'i'), ('OPARG_F', 'f'),
    ('PARAM_DEFAULT', 'f'), ('STATE_DEFAULT', 'f'), ('CAM_I', 'i'), ('CAM_F', 'f'), ('CONS_I', 'i'), ('CONS_F', 'f'),
    ('HULL_F', 'f'),   # reduced convex hulls of mesh collision shapes: per hull its vertices (3 floats each), then its planes (4 each)
]
SECTION_ID = {name: i for i, (name, _) in enumerate(SECTIONS)}
MAGIC = 0x44594742  # 'DYGB'

HDR_I_FIELDS = [
    'nb', 'nl', 'nd', 'ns', 'nv', 'npair', 'ncam', 'nop', 'n_act', 'n_obs', 'n_rew', 'n_term', 'substeps', 'iterations',
    'S', 'P', 'max_contacts', 'nframes', 'hot_start', 'ik_iters', 'ndyn', 'ncons', 'semantics',
    # state offsets
    'S_BPOS', 'S_BQUAT', 'S_BVEL', 'S_BOMEGA', 'S_Q', 'S_QD', 'S_MKP', 'S_MKD', 'S_MTPOS', 'S_MTVEL', 'S_MMAXF',
    'S_MAPPLIED', 'S_JTORQUE', 'S_EXTF', 'S_EXTT', 'S_LPOS', 'S_LQUAT', 'S_LVEL', 'S_LOMEGA', 'S_JREACT', 'S_STEP', 'S_RESETS',
    'S_ADDON',
    # param offsets
    'P_MASS', 'P_INERTIA', 'P_LINDAMP', 'P_ANGDAMP', 'P_JDAMP', 'P_FRICTION', 'P_INITPOSE', 'P_RESTQ', 'P_COLOR',
]
HDR_F_FIELDS = ['dt', 'gx', 'gy', 'gz', 'erp', 'contact_erp', 'linear_slop', 'contact_margin', 'ik_damping',
                'ik_threshold', 'max_joint_vel', 'default_motor_impulse', 'limit_max_impulse', 'ik_null_lambda_sq']

BODY_I_W, BODY_F_W = 8, 8
LINK_I_W, LINK_F_W = 6, 28
SHAPE_I_W, SHAPE_F_W = 8, 20   # ints: body, frame, type, baked, hull vertex offset (floats into HULL_F), vertices, plane offset, planes
VIS_I_W, VIS_F_W = 4, 24
OP_I_W = 8
CAM_I_W, CAM_F_W = 8, 16
CONS_I_W, CONS_F_W = 4, 16

SHAPE_TYPES = {'sphere': 0, 'box': 1, 'capsule': 2, 'cylinder': 3}
JOINT_TYPES = {'fixed': 0, 'revolute': 1, 'continuous': 1, 'prismatic': 2}

OP = dict(JOINT_CTRL=1, EXT_FORCE=2, IK_CTRL=3, JOINT_SENSOR=4, OBJECT_SENSOR=5, REACH_TARGET=6, ELECTRICITY=7,
          STUCK_JOINT=8, TIME_PENALTY=9, EPISODE_TIMER=10, RESPAWN=11, JOINT_RESET=12, DYN_RANDOMIZE=13, ADMITTANCE=14, FT_SENSOR=15,
          FILTERED_WRENCH=16, TILT_TERMINAL=17, VIS_RANDOMIZE=18)
# Ops evaluated by a kernel of their own after the step launches, which the step kernel and the oracle's step skip (they pass over
# op codes they do not know).  Their codes continue the numbering above and are defined beside their kernel, not in
# scene_sections.h: RAY_SENSOR in csrc/dg_ray.cuh (dg_ray_kernel).
KERNEL_OPS = dict(RAY_SENSOR=19)

# Engine semantics that SURVEY Appendix A could only RECALL (no pybullet here to check): each is a named switch of the scene
# header, honoured by the kernels and by the oracle alike, so that the day a pybullet golden vector disagrees the fix is a flag.
# The defaults (all off) are what both arms implemented in round 1.
SEMANTICS = dict(
    wrench_first_substep=1,   # external forces / torques and TORQUE_CONTROL torques act during the first internal sub-step only
                              # (App. A.2 "believed to be cleared after the first substep"); default: during the whole outer step
    motor_clamp_substep=2,    # motor impulse clamp = max force x sub-step dt; default: x fixedTimeStep, the outer dt (App. A.3)
    damping_linear=4,         # multibody velocity damping -m v k only; default: -m v (k + k |v|) (App. A.2)
)

DEFAULT_LATERAL_FRICTION = 0.5
DEFAULT_DAMPING = 0.04  # multibody linear/angular velocity damping (App. A.2)


class BodyInfo:
    """Compile-time view of one spawned model (what `p.getJointInfo` etc. give the reference's add-ons)."""
    def __init__(self, index, name, desc, scale, fixed_base, base_pos, base_quat, mass_override, color):
        self.index, self.name, self.desc, self.scale = index, name, desc, float(scale)
        self.fixed_base = fixed_base
        self.base_pos, self.base_quat = np.asarray(base_pos, float), np.asarray(base_quat, float)
        self.mass_override, self.color = mass_override, color
        self.per_env_pose = False  # set by add-ons (respawn) that move the base per environment
        self.links = desc['links']
        self.n_links = len(self.links) - 1
        self.link_start = self.dof_start = self.frame_base = None  # set by SceneBuilder
        self.joint_dof = []  # per joint index (0..n_links-1): local dof index or -1
        nd = 0
        for l in self.links[1:]:
            if JOINT_TYPES[l['joint']['type']] != 0:
                self.joint_dof.append(nd)
                nd += 1
            else:
                self.joint_dof.append(-1)
        self.n_dofs = nd
        base_mass = self.links[0]['mass'] if mass_override is None else float(mass_override)
        self.base_mass = 0.0 if fixed_base else base_mass
        if self.base_mass == 0.0:
            self.kind = 0 if self.n_links == 0 else 1
        else:
            self.kind = 2

    # --- pybullet-like introspection -------------------------------------------------------------
    def num_joints(self):
        return self.n_links

    def joint_names(self):
        return [l['joint']['name'] for l in self.links[1:]]

    def joint_index(self, name):
        names = self.joint_names()
        return names.index(name) if name in names else -1

    def joint_info(self, i):
        j = self.links[i + 1]['joint']
        movable = self.joint_dof[i] >= 0
        s = self.scale if j['type'] == 'prismatic' else 1.0
        return dict(index=i, name=j['name'], type=j['type'], q_index=(7 + self.joint_dof[i]) if movable else -1,
                    damping=j['damping'], friction=j['friction'], lower=j['lower'] * s, upper=j['upper'] * s,
                    max_force=j['effort'], max_velocity=j['velocity'], link_name=self.links[i + 1]['name'],
                    parent_index=self.links[i + 1]['parent'] - 1)

    def movable_joints(self):
        return [i for i in range(self.n_links) if self.joint_dof[i] >= 0]

    def global_dof(self, joint_index):
        return self.dof_start + self.joint_dof[joint_index]

    def rest_com_pose(self, link_index, joint_angles=None):
        """World pose (Transform) of the COM frame of link `link_index` (-1 = base) at the joint coordinates
        `joint_angles` ({joint index: value}, default all zero): what getBasePositionAndOrientation / getLinkState[0:2]
        report after loadURDF + resetBasePositionAndOrientation + resetJointState."""
        L, s = self.links, self.scale
        q = joint_angles or {}
        LI = [Transform.from_xyz_rpy(np.asarray(l['inertial_xyz']) * s, l['inertial_rpy']) for l in L]
        Tb = Transform(self.base_pos, self.base_quat)
        if link_index < 0:
            return Tb
        chain, k = [], link_index + 1
        while k > 0:
            chain.append(k)
            k = L[k]['parent']
        T = Tb * LI[0].inverse()                      # URDF frame of the base link
        for k in reversed(chain):
            j = L[k]['joint']
            T = T * Transform.from_xyz_rpy(np.asarray(j['xyz']) * s, j['rpy'])
            val = float(q.get(k - 1, 0.0))
            if JOINT_TYPES[j['type']] != 0 and val != 0.0:
                ax = np.asarray(j['axis'], float)
                ax = ax / np.linalg.norm(ax)
                T = T * (Transform((0, 0, 0), np.r_[ax * np.sin(val / 2), np.cos(val / 2)]) if JOINT_TYPES[j['type']] == 1 else Transform(ax * val))
        return T * LI[link_index + 1]

    def frame(self, link_index):
        """Global frame id: base frames come first (one per body), then every link."""
        return self.frame_base if link_index < 0 else self.frame_link0 + link_index


class SceneBuilder:
    def __init__(self, timestep=1 / 240., substeps=2, iterations=150, gravity=(0, 0, -9.81), hot_start=1, max_contacts=16, semantics=(), convex=True):
        self.convex = bool(convex)   # collide mesh links as reduced convex hulls (against boxes and other hulls); False: fitted proxies only
        self.semantics = sum(SEMANTICS[k] for k in semantics)
        self.timestep, self.substeps, self.iterations = float(timestep), int(substeps), int(iterations)
        self.gravity, self.hot_start, self.max_contacts = tuple(float(g) for g in gravity), int(hot_start), int(max_contacts)
        self.bodies = []
        self.ops = []  # (type, iargs, fargs, n_act, n_obs, n_rew, n_term)
        self.cams = []
        self.constraints = []   # fixed constraints between a parent frame and a child frame (model.py:69-77)
        self.addon_state = 0
        self.need_jreact = False   # a force_torque_sensor asks for the joint reaction wrenches (6 floats per link in the state row)
        self.motors_off = []   # global dof indices whose default velocity motor is switched off (admittance_controller.py:34)
        self.finalized = None

    def add_body(self, name, desc, xyz=(0, 0, 0), quat=(0, 0, 0, 1), scale=1.0, fixed_base=False, mass=None, color=None):
        b = BodyInfo(len(self.bodies), name, desc, scale, bool(fixed_base), xyz, quat, mass, color)
        self.bodies.append(b)
        self._assign_indices()
        return b

    def _assign_indices(self):
        nb = len(self.bodies)
        l0 = d0 = 0
        for i, b in enumerate(self.bodies):
            b.link_start, b.dof_start = l0, d0
            b.frame_base = i
            l0 += b.n_links
            d0 += b.n_dofs
        for b in self.bodies:
            b.frame_link0 = nb + b.link_start

    def add_op(self, op, iargs=(), fargs=(), n_act=0, n_obs=0, n_rew=0, n_term=0):
        """Append an add-on op; returns the record so the caller can read the assigned offsets later."""
        rec = dict(type=OP[op] if op in OP else KERNEL_OPS[op], iargs=[int(v) for v in iargs], fargs=[float(v) for v in fargs], n_act=n_act, n_obs=n_obs,
                   n_rew=n_rew, n_term=n_term)
        self.ops.append(rec)
        return rec

    def alloc_addon_state(self, n):
        off = self.addon_state
        self.addon_state += n
        return off

    def add_fixed_constraint(self, body_a, link_a, body_b, link_b, pos_a, quat_a, pos_b=(0, 0, 0), quat_b=(0, 0, 0, 1), max_force=500.0):
        """p.createConstraint(a, link_a, b, link_b, JOINT_FIXED, ..., pos_a, pos_b, quat_a, quat_b): the two joint frames, given
        in the COM frames of the two links (-1 = base), are kept coincident (6 solver rows).  Frames are resolved in finalize()."""
        for b in (body_a, body_b):
            if b.kind == 0:
                b.per_env_pose = True   # keeps a workspace slot for the frame (static bodies are otherwise baked into the tables)
        self.constraints.append(dict(body_a=body_a, link_a=int(link_a), body_b=body_b, link_b=int(link_b), pos_a=list(pos_a),
                                     quat_a=list(quat_a), pos_b=list(pos_b), quat_b=list(quat_b), max_force=float(max_force)))
        return len(self.constraints) - 1

    def add_camera(self, frame, xyz, quat, width, height, fov, near, far):
        rec = dict(frame=int(frame), xyz=list(xyz), quat=list(quat), width=int(width), height=int(height), fov=float(fov),
                   near=float(near), far=float(far))
        self.cams.append(rec)
        return len(self.cams) - 1

    # ---------------------------------------------------------------------------------------------
    def finalize(self):
        self._assign_indices()
        B = self.bodies
        nb = len(B)
        nl = sum(b.n_links for b in B)
        nd = sum(b.n_dofs for b in B)
        nframes = nb + nl

        body_i = np.zeros((nb, BODY_I_W), np.int32)
        body_f = np.zeros((nb, BODY_F_W))
        link_i = np.zeros((max(nl, 0), LINK_I_W), np.int32)
        link_f = np.zeros((max(nl, 0), LINK_F_W))
        mass = np.zeros(nframes)
        inertia = np.zeros((nframes, 3))
        jdamp = np.zeros(nd)
        restq = np.zeros(nd)
        init_pose = np.zeros((nb, 7))
        shapes, visuals = [], []
        frame_movable = np.zeros(nframes, bool)

        dyn_index, ndyn = {}, 0
        for b in B:
            dyn_index[b.index] = ndyn if b.kind != 0 else -1
            ndyn += int(b.kind != 0)
        for b in B:
            s = b.scale
            L = b.links
            LI = [Transform.from_xyz_rpy(np.asarray(l['inertial_xyz']) * s, l['inertial_rpy']) for l in L]
            baked = int(b.kind == 0 and not b.per_env_pose)
            body_i[b.index] = [b.kind, b.link_start, b.n_links, b.dof_start, b.n_dofs, b.frame_link0, dyn_index[b.index], baked]
            body_f[b.index, 0:3] = LI[0].p
            body_f[b.index, 3:7] = LI[0].q
            init_pose[b.index, 0:3] = b.base_pos
            init_pose[b.index, 3:7] = b.base_quat
            mass[b.frame_base] = b.base_mass
            inertia[b.frame_base] = inertia_from_rule(L[0]['inertia_rule'], b.base_mass, s, L[0]['inertia_xml'])
            frame_movable[b.frame_base] = b.kind == 2
            for k in range(1, len(L)):
                l = L[k]
                j = l['joint']
                gl = b.link_start + k - 1
                fr = b.frame_link0 + k - 1
                jt = JOINT_TYPES[j['type']]
                parent_local = l['parent']  # index into L (0 = base)
                parent_global = -1 if parent_local == 0 else b.link_start + parent_local - 1
                dof = b.dof_start + b.joint_dof[k - 1] if jt != 0 else -1
                has_limit = int(j['type'] in ('revolute', 'prismatic') and j['lower'] <= j['upper'])
                link_i[gl] = [b.index, parent_global, jt, dof, has_limit, 0]
                p2j = Transform.from_xyz_rpy(np.asarray(j['xyz']) * s, j['rpy'])
                offA = LI[parent_local].inverse() * p2j
                T0 = offA * LI[k]
                axis = np.asarray(j['axis'], float)
                n = np.linalg.norm(axis)
                axis = axis / n if n > 0 else np.array([1.0, 0, 0])
                a = quat_rotate(quat_conj(LI[k].q), axis)
                d = quat_rotate(quat_conj(LI[k].q), LI[k].p)
                ls = s if jt == 2 else 1.0
                link_f[gl, 0:4] = T0.q
                link_f[gl, 4:7] = offA.p
                link_f[gl, 7:10] = d
                link_f[gl, 10:13] = a
                link_f[gl, 13:16] = LI[k].p
                link_f[gl, 16:20] = LI[k].q
                link_f[gl, 20:25] = [j['lower'] * ls, j['upper'] * ls, j['effort'], j['velocity'], j['friction']]
                mass[fr] = l['mass']
                inertia[fr] = inertia_from_rule(l['inertia_rule'], l['mass'], s, l['inertia_xml'])
                pm = frame_movable[b.frame_base] if parent_local == 0 else frame_movable[b.frame_link0 + parent_local - 1]
                frame_movable[fr] = pm or jt != 0
                if jt != 0:
                    jdamp[dof] = j['damping']
            for k, l in enumerate(L):
                fr = b.frame(k - 1)
                fric = l['lateral_friction'] if l['lateral_friction'] is not None else DEFAULT_LATERAL_FRICTION
                Tci = LI[k].inverse()
                for c in l['collisions']:
                    T = Tci * Transform(np.asarray(c['xyz']) * s, c['quat'])
                    dims = np.asarray(c['dims'], float) * s
                    Tw = Transform(b.base_pos, b.base_quat) * T
                    shapes.append(dict(body=b.index, frame=fr, type=SHAPE_TYPES[c['type']], pos=T.p, quat=T.q, dims=dims,
                                       friction=fric, baked=int(b.kind == 0 and not b.per_env_pose), wpos=Tw.p, wquat=Tw.q,
                                       hull=c.get('hull') if self.convex else None, scale=s))
                for v in l['visuals']:
                    T = Tci * Transform(np.asarray(v['xyz']) * s, v['quat'])
                    dims = np.asarray(v['dims'], float) * s
                    rgba = list(v.get('rgba', [1, 1, 1, 1]))
                    if b.color is not None and k == 0:
                        rgba = [float(x) for x in b.color]
                    Tw = Transform(b.base_pos, b.base_quat) * T
                    visuals.append(dict(body=b.index, frame=fr, type=SHAPE_TYPES[v['type']], pos=T.p, quat=T.q, dims=dims, rgba=rgba,
                                        baked=int(b.kind == 0 and not b.per_env_pose), wpos=Tw.p, wquat=Tw.q))

        ns, nv = len(shapes), len(visuals)
        shape_i = np.zeros((ns, SHAPE_I_W), np.int32)
        hull_f = []
        shape_f = np.zeros((ns, SHAPE_F_W))
        friction = np.zeros(ns)
        for i, sh in enumerate(shapes):
            shape_i[i, :4] = [sh['body'], sh['frame'], sh['type'], sh['baked']]
            shape_f[i, 12:15], shape_f[i, 15:19] = sh['wpos'], sh['wquat']
            shape_f[i, 0:3], shape_f[i, 3:7], shape_f[i, 7:11] = sh['pos'], sh['quat'], sh['dims']
            d = sh['dims']
            shape_f[i, 11] = {0: d[0], 1: float(np.linalg.norm(d[:3])), 2: d[0] + d[1], 3: float(np.hypot(d[0], d[1]))}[sh['type']]
            friction[i] = sh['friction']
            if sh.get('hull'):   # reduced convex hull of a mesh link, in the shape frame, scaled like the model
                V = np.asarray(sh['hull']['verts'], float) * sh['scale']
                Pl = np.asarray(sh['hull']['planes'], float).copy()
                Pl[:, 3] *= sh['scale']
                shape_i[i, 4:8] = [len(hull_f), len(V), len(hull_f) + 3 * len(V), len(Pl)]
                hull_f += V.reshape(-1).tolist() + Pl.reshape(-1).tolist()
                shape_f[i, 11] = max(shape_f[i, 11], float(np.linalg.norm(V, axis=1).max()))   # the bound the broad phase uses covers the hull
        vis_i = np.zeros((nv, VIS_I_W), np.int32)
        vis_f = np.zeros((nv, VIS_F_W))
        for i, v in enumerate(visuals):
            vis_i[i] = [v['frame'], v['type'], v['baked'], v['body']]   # body index = the uid pybullet's segmentation mask reports
            vis_f[i, 16:19], vis_f[i, 19:23] = v['wpos'], v['wquat']
            vis_f[i, 0:3], vis_f[i, 3:7], vis_f[i, 7:11], vis_f[i, 11:15] = v['pos'], v['quat'], v['dims'], v['rgba']
            d = v['dims']
            vis_f[i, 15] = {0: d[0], 1: float(np.linalg.norm(d[:3])), 2: d[0] + d[1], 3: float(np.hypot(d[0], d[1]))}[v['type']]

        pairs = []
        for i in range(ns):
            for j in range(i + 1, ns):
                if shapes[i]['body'] == shapes[j]['body']:
                    continue
                if not (frame_movable[shapes[i]['frame']] or frame_movable[shapes[j]['frame']]):
                    continue
                pairs.append((i, j))
        pair_i = np.array(pairs, np.int32).reshape(-1, 2)

        # ---- layouts ------------------------------------------------------------------------------
        lay = OrderedDict()
        off = 0
        for name, n in [('S_BPOS', 3 * nb), ('S_BQUAT', 4 * nb), ('S_BVEL', 3 * nb), ('S_BOMEGA', 3 * nb), ('S_Q', nd),
                        ('S_QD', nd), ('S_MKP', nd), ('S_MKD', nd), ('S_MTPOS', nd), ('S_MTVEL', nd), ('S_MMAXF', nd),
                        ('S_MAPPLIED', nd), ('S_JTORQUE', nd), ('S_EXTF', 3 * nframes), ('S_EXTT', 3 * nframes),
                        ('S_LPOS', 3 * nl), ('S_LQUAT', 4 * nl), ('S_LVEL', 3 * nl), ('S_LOMEGA', 3 * nl),
                        ('S_JREACT', 6 * nl if self.need_jreact else 0), ('S_STEP', 1),
                        ('S_RESETS', 1), ('S_ADDON', self.addon_state)]:
            lay[name] = off
            off += n
        S = off
        off = 0
        for name, n in [('P_MASS', nframes), ('P_INERTIA', 3 * nframes), ('P_LINDAMP', nb), ('P_ANGDAMP', nb), ('P_JDAMP', nd),
                        ('P_FRICTION', ns), ('P_INITPOSE', 7 * nb), ('P_RESTQ', nd), ('P_COLOR', 3 * nv)]:   # P_COLOR: rgb per visual shape (visual_randomizer)
            lay[name] = off
            off += n
        P = off

        param = np.zeros(P)
        param[lay['P_MASS']:lay['P_MASS'] + nframes] = mass
        param[lay['P_INERTIA']:lay['P_INERTIA'] + 3 * nframes] = inertia.reshape(-1)
        param[lay['P_LINDAMP']:lay['P_LINDAMP'] + nb] = DEFAULT_DAMPING
        param[lay['P_ANGDAMP']:lay['P_ANGDAMP'] + nb] = DEFAULT_DAMPING
        param[lay['P_JDAMP']:lay['P_JDAMP'] + nd] = jdamp
        param[lay['P_FRICTION']:lay['P_FRICTION'] + ns] = friction
        param[lay['P_INITPOSE']:lay['P_INITPOSE'] + 7 * nb] = init_pose.reshape(-1)
        param[lay['P_RESTQ']:lay['P_RESTQ'] + nd] = restq
        param[lay['P_COLOR']:lay['P_COLOR'] + 3 * nv] = vis_f[:, 11:14].reshape(-1)

        state = np.zeros(S)
        state[lay['S_BPOS']:lay['S_BPOS'] + 3 * nb] = init_pose[:, 0:3].reshape(-1)
        state[lay['S_BQUAT']:lay['S_BQUAT'] + 4 * nb] = init_pose[:, 3:7].reshape(-1)
        # default velocity motor on every 1-DoF joint: target 0, kd 1, max impulse 1 per solve (App. A.3)
        dt = self.timestep
        state[lay['S_MKD']:lay['S_MKD'] + nd] = 1.0
        state[lay['S_MMAXF']:lay['S_MMAXF'] + nd] = 1.0 / dt
        for d in self.motors_off:
            state[lay['S_MMAXF'] + d] = 0.0
        state[lay['S_LQUAT'] + 3:lay['S_LQUAT'] + 4 * nl:4] = 1.0

        # ---- ops ----------------------------------------------------------------------------------
        nop = len(self.ops)
        # the per-step action mask (dg_set_action_mask: add-ons absent from the action dict are not updated, diy_gym.py:202-204)
        # has 128 bits: an action-bearing op beyond them could not be switched off
        for k, op in enumerate(self.ops):
            if k >= 128 and op['n_act']:
                raise ValueError('more than 128 add-on ops before an action-bearing one (op %d): the action mask has 128 bits' % k)
        op_i = np.zeros((nop, OP_I_W), np.int32)
        oparg_i, oparg_f = [], []
        n_act = n_obs = n_rew = n_term = 0
        for k, o in enumerate(self.ops):
            o['act_off'], o['obs_off'], o['rew_off'], o['term_off'] = n_act, n_obs, n_rew, n_term
            op_i[k] = [o['type'], len(oparg_i), len(oparg_f), n_act if o['n_act'] else -1, n_obs if o['n_obs'] else -1,
                       n_rew if o['n_rew'] else -1, n_term if o['n_term'] else -1, 0]
            oparg_i += o['iargs']
            oparg_f += o['fargs']
            n_act += o['n_act']
            n_obs += o['n_obs']
            n_rew += o['n_rew']
            n_term += o['n_term']

        ncam = len(self.cams)
        ncons = len(self.constraints)
        cons_i = np.zeros((ncons, CONS_I_W), np.int32)
        cons_f = np.zeros((ncons, CONS_F_W))
        for k, c in enumerate(self.constraints):
            cons_i[k, 0:2] = [c['body_a'].frame(c['link_a']), c['body_b'].frame(c['link_b'])]
            cons_f[k, 0:3], cons_f[k, 3:7], cons_f[k, 7:10], cons_f[k, 10:14], cons_f[k, 14] = c['pos_a'], c['quat_a'], c['pos_b'], c['quat_b'], c['max_force']
        cam_i = np.zeros((ncam, CAM_I_W), np.int32)
        cam_f = np.zeros((ncam, CAM_F_W))
        for k, c in enumerate(self.cams):
            cam_i[k, :3] = [c['frame'], c['width'], c['height']]
            cam_f[k, 0:3], cam_f[k, 3:7] = c['xyz'], c['quat']
            cam_f[k, 7:10] = [c['fov'], c['near'], c['far']]

        # contact-point capacity per environment (extension key `max_contacts`): floating bodies rest on several
        # points at once, fixed-base arms only touch occasionally - their scenes keep the solver workspace small
        if self.max_contacts <= 0:
            self.max_contacts = 16 if any(b.kind == 2 for b in B) else 8
        if self.max_contacts > 21:
            raise ValueError('max_contacts is limited to 21 (the solver tracks at most 63 contact rows per environment)')
        hdr = dict(nb=nb, nl=nl, nd=nd, ns=ns, nv=nv, npair=len(pairs), ncam=ncam, nop=nop, n_act=n_act, n_obs=n_obs,
                   n_rew=n_rew, n_term=n_term, substeps=self.substeps, iterations=self.iterations, S=S, P=P,
                   max_contacts=self.max_contacts, nframes=nframes, hot_start=self.hot_start, ik_iters=20, ndyn=ndyn, ncons=ncons, semantics=self.semantics)
        hdr.update(lay)
        hdr_i = np.array([hdr[k] for k in HDR_I_FIELDS], np.int32)
        hf = dict(dt=self.timestep, gx=self.gravity[0], gy=self.gravity[1], gz=self.gravity[2], erp=0.2, contact_erp=0.2,
                  linear_slop=0.0, contact_margin=0.0, ik_damping=0.5, ik_threshold=1e-4, max_joint_vel=100.0,
                  default_motor_impulse=1.0, limit_max_impulse=100.0, ik_null_lambda_sq=0.36)
        hdr_f = np.array([hf[k] for k in HDR_F_FIELDS])

        sec = dict(HDR_I=hdr_i, HDR_F=hdr_f, BODY_I=body_i, BODY_F=body_f, LINK_I=link_i, LINK_F=link_f, SHAPE_I=shape_i,
                   SHAPE_F=shape_f, PAIR_I=pair_i, VIS_I=vis_i, VIS_F=vis_f, OP_I=op_i, OPARG_I=np.array(oparg_i, np.int32),
                   OPARG_F=np.array(oparg_f, float), PARAM_DEFAULT=param, STATE_DEFAULT=state, CAM_I=cam_i, CAM_F=cam_f, CONS_I=cons_i, CONS_F=cons_f,
                   HULL_F=np.array(hull_f, float))
        self.finalized = Scene(sec, hdr, hf, self)
        return self.finalized


class Scene:
    """Finalised scene: named sections, header dict, and the packed (ibuf, fbuf) pair."""
    def __init__(self, sections, hdr, hdr_f, builder):
        self.sec, self.hdr, self.hdr_f, self.builder = sections, hdr, hdr_f, builder
        self.bodies = builder.bodies
        ints, floats = [], []
        ioff = 2 + 3 * len(SECTIONS)
        foff = 0
        table = []
        for name, kind in SECTIONS:
            arr = np.ascontiguousarray(sections[name]).reshape(-1)
            if kind == 'i':
                table += [0, ioff, arr.size]
                ints.append(arr.astype(np.int32))
                ioff += arr.size
            else:
                table += [1, foff, arr.size]
                floats.append(arr.astype(np.float64))
                foff += arr.size
        self.ibuf = np.concatenate([np.array([MAGIC, len(SECTIONS)] + table, np.int32)] + ints).astype(np.int32)
        self.fbuf = np.concatenate(floats).astype(np.float64) if floats else np.zeros(0)

    def __getitem__(self, k):
        return self.hdr[k]

    def state_slice(self, name, n):
        return slice(self.hdr[name], self.hdr[name] + n)


def write_c_headers():
    """Regenerates the two copies of scene_sections.h (csrc/ for the kernels, oracle/ for the checker)."""
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    for dst in (os.path.join(here, '..', 'csrc', 'scene_sections.h'), os.path.join(here, '..', '..', 'oracle', 'scene_sections.h')):
        with open(dst, 'w') as f:
            f.write(emit_c_header())


def emit_c_header():
    """Text of `scene_sections.h` (generated into oracle/ and csrc/; data layout only, no algorithm)."""
    out = ['/* GENERATED by diy_gym_b200/compiler/scene.py:emit_c_header - scene buffer layout (data only). */',
           '#ifndef DG_SCENE_SECTIONS_H', '#define DG_SCENE_SECTIONS_H', '#define DG_SCENE_MAGIC 0x%X' % MAGIC,
           '#define DG_NSECTIONS %d' % len(SECTIONS)]
    for i, (name, _) in enumerate(SECTIONS):
        out.append('#define SEC_%s %d' % (name, i))
    for i, name in enumerate(HDR_I_FIELDS):
        out.append('#define HI_%s %d' % (name, i))
    for i, name in enumerate(HDR_F_FIELDS):
        out.append('#define HF_%s %d' % (name, i))
    for k, v in [('BODY_I_W', BODY_I_W), ('BODY_F_W', BODY_F_W), ('LINK_I_W', LINK_I_W), ('LINK_F_W', LINK_F_W),
                 ('SHAPE_I_W', SHAPE_I_W), ('SHAPE_F_W', SHAPE_F_W), ('VIS_I_W', VIS_I_W), ('VIS_F_W', VIS_F_W),
                 ('OP_I_W', OP_I_W), ('CAM_I_W', CAM_I_W), ('CAM_F_W', CAM_F_W), ('CONS_I_W', CONS_I_W), ('CONS_F_W', CONS_F_W)]:
        out.append('#define DG_%s %d' % (k, v))
    for k, v in OP.items():
        out.append('#define OP_%s %d' % (k, v))
    for k, v in SEMANTICS.items():
        out.append('#define SEM_%s %d' % (k.upper(), v))
    for k, v in SHAPE_TYPES.items():
        out.append('#define SHAPE_%s %d' % (k.upper(), v))
    out.append('#endif')
    return '\n'.join(out) + '\n'
