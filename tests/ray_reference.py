"""fp64 reference of the ray_sensor op (test infrastructure): pybullet's rayTestBatch against the collision shapes of a compiled
scene, restated in numpy from the scene tables and a state row, independently of the fp32 routines in csrc/dg_ray.cuh.

Semantics (DESIGN.md section 2): per ray the distance to the first surface the ray enters with t in (min, max] (max on a miss) and
the body index hit (-1 on a miss).  The ray starts at min; a shape that contains that point is not reported.  Mesh shapes with a
reduced convex hull (SHAPE_I[5] > 0) are their hull (Cyrus-Beck clip against the HULL_F planes); the rest are their primitive.
Shape poses: the compiled world pose of baked shapes (SHAPE_F[12:19]), else the COM pose of the frame in the state row's link
cache times the shape's local pose.  Sensor pose: the frame's URDF link pose (the camera's convention) times xyz / quat."""
import numpy as np

from diy_gym_b200.compiler.mathutil import quat_to_mat
from diy_gym_b200.compiler.scene import KERNEL_OPS

SPHERE, BOX, CAPSULE, CYLINDER = 0, 1, 2, 3
EPS = 1e-9


def frame_com_pose(scene, st, f):
    h, nb = scene.hdr, scene.hdr['nb']
    if f < nb:
        return quat_to_mat(st[h['S_BQUAT'] + 4 * f:h['S_BQUAT'] + 4 * f + 4]), st[h['S_BPOS'] + 3 * f:h['S_BPOS'] + 3 * f + 3].copy()
    gl = f - nb
    return quat_to_mat(st[h['S_LQUAT'] + 4 * gl:h['S_LQUAT'] + 4 * gl + 4]), st[h['S_LPOS'] + 3 * gl:h['S_LPOS'] + 3 * gl + 3].copy()


def frame_link_pose(scene, st, f):
    """URDF link frame = COM frame times the inverse of the link's inertial frame (LINK_F[16:20] its rotation, [7:10] its offset
    in the COM frame)."""
    R, p = frame_com_pose(scene, st, f)
    if f >= scene.hdr['nb']:
        lf = scene.sec['LINK_F'][f - scene.hdr['nb']]
        p = p - R @ lf[7:10]
        R = R @ quat_to_mat(lf[16:20]).T
    return R, p


def shape_poses(scene, st):
    SI, SF = scene.sec['SHAPE_I'], scene.sec['SHAPE_F']
    out = []
    for s in range(len(SI)):
        if SI[s, 3]:
            out.append((quat_to_mat(SF[s, 15:19]), SF[s, 12:15].copy()))
        else:
            Rf, pf = frame_com_pose(scene, st, int(SI[s, 1]))
            out.append((Rf @ quat_to_mat(SF[s, 3:7]), pf + Rf @ SF[s, 0:3]))
    return out


def _inside(kind, d, planes, o):
    if planes is not None:
        return np.all(o @ planes[:, :3].T - planes[:, 3] <= 0, axis=1)
    if kind == SPHERE:
        return np.sum(o * o, axis=1) <= d[0] ** 2
    if kind == BOX:
        return np.all(np.abs(o) <= d[:3], axis=1)
    r2 = o[:, 0] ** 2 + o[:, 1] ** 2
    if kind == CYLINDER:
        return (r2 <= d[0] ** 2) & (np.abs(o[:, 2]) <= d[1])
    dz = o[:, 2] - np.clip(o[:, 2], -d[1], d[1])
    return r2 + dz * dz <= d[0] ** 2


def _entry(kind, d, planes, o, u):
    """Nearest entry parameter (> EPS) of the rays o + t u into the shape, inf where there is none."""
    n = len(o)
    best = np.full(n, np.inf)
    with np.errstate(divide='ignore', invalid='ignore'):
        if planes is not None:
            te, tx, ok = np.full(n, -np.inf), np.full(n, np.inf), np.ones(n, bool)
            for q in planes:
                den, num = u @ q[:3], q[3] - o @ q[:3]
                par = np.abs(den) < 1e-18
                ok &= ~(par & (num < 0))
                t = np.where(par, 0.0, num / np.where(par, 1.0, den))
                te = np.where(~par & (den < 0), np.maximum(te, t), te)
                tx = np.where(~par & (den > 0), np.minimum(tx, t), tx)
            hit = ok & (te <= tx) & (te > EPS)
            return np.where(hit, te, np.inf)
        cands = []
        if kind in (SPHERE, CAPSULE):
            for cz in ([0.0] if kind == SPHERE else [-d[1], d[1]]):
                oc = o - [0, 0, cz]
                A, B, C = np.sum(u * u, axis=1), np.sum(oc * u, axis=1), np.sum(oc * oc, axis=1) - d[0] ** 2
                disc = B * B - A * C
                cands.append(np.where(disc >= 0, (-B - np.sqrt(np.maximum(disc, 0))) / A, np.inf))
        if kind in (CAPSULE, CYLINDER):
            A = u[:, 0] ** 2 + u[:, 1] ** 2
            B = o[:, 0] * u[:, 0] + o[:, 1] * u[:, 1]
            C = o[:, 0] ** 2 + o[:, 1] ** 2 - d[0] ** 2
            disc = B * B - A * C
            t = (-B - np.sqrt(np.maximum(disc, 0))) / np.where(A > 1e-18, A, 1.0)
            z = o[:, 2] + t * u[:, 2]
            cands.append(np.where((A > 1e-18) & (disc >= 0) & (np.abs(z) <= d[1]), t, np.inf))
            if kind == CYLINDER:
                nz = np.abs(u[:, 2]) > 1e-18
                for s in (-1.0, 1.0):
                    t = (s * d[1] - o[:, 2]) / np.where(nz, u[:, 2], 1.0)
                    x, y = o[:, 0] + t * u[:, 0], o[:, 1] + t * u[:, 1]
                    cands.append(np.where(nz & (x * x + y * y <= d[0] ** 2), t, np.inf))
        if kind == BOX:
            t0, t1 = np.full(n, -np.inf), np.full(n, np.inf)
            for i in range(3):
                par = np.abs(u[:, i]) < 1e-18
                ins = np.abs(o[:, i]) <= d[i]
                ui = np.where(par, 1.0, u[:, i])
                ta, tb = (-d[i] - o[:, i]) / ui, (d[i] - o[:, i]) / ui
                lo, hi = np.minimum(ta, tb), np.maximum(ta, tb)
                lo = np.where(par, np.where(ins, -np.inf, np.inf), lo)
                hi = np.where(par, np.where(ins, np.inf, -np.inf), hi)
                t0, t1 = np.maximum(t0, lo), np.minimum(t1, hi)
            cands.append(np.where(t0 <= t1, t0, np.inf))
        for t in cands:
            best = np.where((t > EPS) & (t < best), t, best)
    return best


def cast(scene, st):
    """Observation row [n_obs] (fp64) with the slices of every ray_sensor op filled from the state row `st`; other slices are 0."""
    st = np.asarray(st, np.float64)
    SI, SF, H = scene.sec['SHAPE_I'], scene.sec['SHAPE_F'], scene.sec['HULL_F']
    poses = shape_poses(scene, st)
    obs = np.zeros(scene.hdr['n_obs'])
    for op in scene.builder.ops:
        if op['type'] != KERNEL_OPS['RAY_SENSOR']:
            continue
        frame, nr, flags = op['iargs']
        fa = np.asarray(op['fargs'])
        Rp, pp = frame_link_pose(scene, st, frame) if frame >= 0 else (np.eye(3), np.zeros(3))
        Rs, ps = Rp @ quat_to_mat(fa[3:7]), pp + Rp @ fa[0:3]
        tmin, tmax = fa[7], fa[8]
        D = fa[9:9 + 3 * nr].reshape(nr, 3) @ Rs.T
        start = ps + tmin * D
        best, body = np.full(nr, tmax - tmin), np.full(nr, -1.0)
        for s in range(len(SI)):
            R, p = poses[s]
            o, u = (start - p) @ R, D @ R   # shape frame
            planes = H[SI[s, 6]:SI[s, 6] + 4 * SI[s, 7]].reshape(-1, 4) if SI[s, 5] > 0 else None
            t = _entry(int(SI[s, 2]), SF[s, 7:11], planes, o, u)
            hit = ~_inside(int(SI[s, 2]), SF[s, 7:11], planes, o) & (t < best)
            best, body = np.where(hit, t, best), np.where(hit, float(SI[s, 0]), body)
        off = op['obs_off']
        obs[off:off + nr] = np.where(body >= 0, tmin + best, tmax)
        if flags & 1:
            obs[off + nr:off + 2 * nr] = body
    return obs
