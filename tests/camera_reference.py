"""fp64 reference of the camera (test infrastructure): dgo_render_seg (oracle/bullet_restatement.c) restated in numpy, vectorised
over the pixels, independently of dg_render_kernel and of the oracle's code.

It reads the scene tables, one state row and one parameter row.  Poses: the compiled world pose of baked visuals (VIS_F[16:23],
what the kernel reads through vis_wb), else the COM pose of the frame in the state row's link cache times the visual's local pose;
the camera sits on the URDF link frame of its frame (or in the world) times its xyz / quat.  Per pixel the ray
eye + t R_cam ((i + 0.5) / W * 2 - 1) tan(fov / 2) aspect, (1 - (j + 0.5) / H * 2) tan(fov / 2), -1)  (t = eye-space depth) is cast
against every visual shape:
  - a shape's hit is its nearest entry with t > 1e-9 (ray_shape: spheres / capsule end spheres, then the side of capsules and
    cylinders, then cylinder caps, then box slabs, a later candidate replacing an earlier one only when strictly nearer); the caps
    of a cylinder are hit from inside, so a camera inside a cylinder sees the far cap;
  - a shape whose hit has t < near is not seen at all, and only t < far counts;
  - the nearest shape wins, the first in index order on an exact tie;
  - colour = P_COLOR of the shape x (0.4 + 0.6 max(n . light, 0)), depth = -t, mask = the shape's body; background rgb 1,
    depth -far, mask -1.

`render` also returns where an fp32 renderer may rightly differ (the ambiguity mask) and which mask values it may then show."""
import numpy as np

from diy_gym_b200.compiler.mathutil import quat_to_mat
from tests.ray_reference import BOX, CAPSULE, CYLINDER, EPS, SPHERE, frame_com_pose, frame_link_pose

LIGHT = np.array([0.4082482904638631, 0.4082482904638631, 0.8164965809277261])
JITTER = 1e-3        # pixels: a result that changes within this shift of the ray is a silhouette / seam pixel
NEAR_TOL = 1e-5      # relative: an entry this close to the near or far plane may fall either side of it in fp32
TIE_TOL = 1e-6       # relative: two shapes entered this close to each other may swap in fp32
# fp32 rounding of the eye, the ray direction and the shape poses turns a ray by well under RAY_EPS radians; where turning it by
# that much would change depth (relative) or colour by more than COND_DEPTH / COND_RGB, judged from the JITTER shift, the hit is
# grazing and an fp32 renderer may be off by more than its usual error
RAY_EPS = 1e-6
COND_DEPTH = 2e-5
COND_RGB = 1e-4
U32 = 2.0 ** -24     # unit roundoff of fp32


def visual_poses(scene, st):
    VI, VF = scene.sec['VIS_I'], scene.sec['VIS_F']
    out = []
    for s in range(len(VI)):
        if VI[s, 2]:
            out.append((quat_to_mat(VF[s, 19:23]), VF[s, 16:19].copy()))
        else:
            Rf, pf = frame_com_pose(scene, st, int(VI[s, 0]))
            out.append((Rf @ quat_to_mat(VF[s, 3:7]), pf + Rf @ VF[s, 0:3]))
    return out


def camera_pose(scene, st, cam):
    ci, cf = scene.sec['CAM_I'][cam], scene.sec['CAM_F'][cam]
    Rp, pp = frame_link_pose(scene, st, int(ci[0])) if ci[0] >= 0 else (np.eye(3), np.zeros(3))
    return Rp @ quat_to_mat(cf[3:7]), pp + Rp @ cf[0:3]


def pixel_directions(scene, cam, dx=0.0, dy=0.0):
    """Camera-space ray directions [H * W, 3] (z = -1), row-major pixels, shifted by (dx, dy) pixels."""
    w, h = int(scene.sec['CAM_I'][cam][1]), int(scene.sec['CAM_I'][cam][2])
    th = np.tan(scene.sec['CAM_F'][cam][7] * np.pi / 360.0)
    j, i = np.meshgrid(np.arange(h, dtype=float), np.arange(w, dtype=float), indexing='ij')
    x = ((i.ravel() + 0.5 + dx) / w * 2 - 1) * th * (w / h)
    y = (1 - (j.ravel() + 0.5 + dy) / h * 2) * th
    return np.stack([x, y, -np.ones_like(x)], axis=1)


def entry(kind, d, o, u):
    """The oracle's ray_shape without tmax: nearest entry t > 1e-9 of the rays o + t u (shape frame; o [3], u [n, 3]), its
    shape-frame normal and the surface piece it lies on (0 / 1 capsule end spheres or the sphere, 2 side, 3 / 4 cylinder caps,
    5 + 2 axis + (normal > 0) box faces).  t = inf and piece -1 where there is none.

    Also the size of one fp32 rounding error of t and of the normal for the same arithmetic: a sphere, capsule or cylinder side
    solves A t^2 + 2 B t + C = 0, whose discriminant B^2 - A C cancels, so one ulp of its terms moves t by
    U32 (B^2 + |A C|) / (A sqrt(disc)) and the normal (o + t u) / r by that times |u| / r; planes (caps, box faces) only round
    t by an ulp of |o| / |u| and have exact normals."""
    n = len(u)
    best, nrm, piece = np.full(n, np.inf), np.tile([0.0, 0.0, 1.0], (n, 1)), np.full(n, -1)
    terr, nerr = np.zeros(n), np.zeros(n)
    ulen = np.sqrt(np.sum(u * u, axis=1))

    def take(t, nn, pc, te, ne=0.0):
        upd = (t > EPS) & (t < best)
        best[upd] = t[upd]
        nrm[upd] = nn[upd]
        piece[upd] = pc[upd] if np.ndim(pc) else pc
        terr[upd] = te[upd]
        nerr[upd] = ne[upd] if np.ndim(ne) else ne

    def quadric_err(A, B, C, disc, olen, r):
        te = U32 * (B * B + np.abs(A * C)) / (A * np.sqrt(np.maximum(disc, 1e-300)))
        return te, (te * ulen + U32 * olen) / r

    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        if kind in (SPHERE, CAPSULE):
            for k, cz in enumerate([0.0] if kind == SPHERE else [-d[1], d[1]]):
                oc = o - np.array([0.0, 0.0, cz])
                A, B, C = np.sum(u * u, axis=1), u @ oc, oc @ oc - d[0] * d[0]
                disc = B * B - A * C
                t = np.where(disc >= 0, (-B - np.sqrt(np.maximum(disc, 0))) / A, np.nan)
                take(t, (oc + t[:, None] * u) / d[0], k, *quadric_err(A, B, C, disc, np.linalg.norm(oc), d[0]))
        if kind in (CAPSULE, CYLINDER):
            A = u[:, 0] ** 2 + u[:, 1] ** 2
            B = o[0] * u[:, 0] + o[1] * u[:, 1]
            C = o[0] ** 2 + o[1] ** 2 - d[0] ** 2
            disc = B * B - A * C
            ok = (A > 1e-18) & (disc >= 0)
            t = np.where(ok, (-B - np.sqrt(np.maximum(disc, 0))) / np.where(ok, A, 1.0), np.nan)
            z = o[2] + t * u[:, 2]
            t = np.where(np.abs(z) <= d[1], t, np.nan)
            nn = np.stack([(o[0] + t * u[:, 0]) / d[0], (o[1] + t * u[:, 1]) / d[0], np.zeros(n)], axis=1)
            take(t, nn, 2, *quadric_err(np.where(ok, A, 1.0), B, C, disc, np.hypot(o[0], o[1]), d[0]))
            if kind == CYLINDER:
                nz = np.abs(u[:, 2]) > 1e-18
                for s in (-1.0, 1.0):
                    t = np.where(nz, (s * d[1] - o[2]) / np.where(nz, u[:, 2], 1.0), np.nan)
                    x, y = o[0] + t * u[:, 0], o[1] + t * u[:, 1]
                    t = np.where(x * x + y * y <= d[0] * d[0], t, np.nan)
                    take(t, np.tile([0.0, 0.0, s], (n, 1)), 3 if s < 0 else 4, U32 * np.linalg.norm(o) / ulen)
        if kind == BOX:
            t0, t1 = np.full(n, -1e300), np.full(n, 1e300)
            ax0, sg0, miss = np.zeros(n, int), np.ones(n), np.zeros(n, bool)
            for i in range(3):
                par = np.abs(u[:, i]) < 1e-18
                miss |= par & (abs(o[i]) > d[i])
                ui = np.where(par, 1.0, u[:, i])
                ta, tb = (-d[i] - o[i]) / ui, (d[i] - o[i]) / ui
                sg = np.where(ta > tb, 1.0, -1.0)
                ta, tb = np.minimum(ta, tb), np.maximum(ta, tb)
                up = ~par & (ta > t0)
                t0, ax0, sg0 = np.where(up, ta, t0), np.where(up, i, ax0), np.where(up, sg, sg0)
                t1 = np.where(par, t1, np.minimum(t1, tb))
            t = np.where(~miss & (t0 <= t1), t0, np.nan)
            nn = np.zeros((n, 3))
            nn[np.arange(n), ax0] = sg0
            take(t, nn, 5 + 2 * ax0 + (sg0 > 0), U32 * np.linalg.norm(o) / ulen)
    return best, nrm, piece, terr, nerr


def cast(scene, st, prm, cam, dx=0.0, dy=0.0, keep_entries=False):
    """One ray per pixel: the hit visual per pixel (-1: none), its depth t, colour and surface piece; with keep_entries also
    every shape's entry T [nv, npx] (inf: none) and the distance |eye - shape centre| per shape.  t_err / rgb_err: one fp32
    rounding error of the hit's depth and colour (entry())."""
    VI, VF, h = scene.sec['VIS_I'], scene.sec['VIS_F'], scene.hdr
    nv = len(VI)
    near, far = scene.sec['CAM_F'][cam][8], scene.sec['CAM_F'][cam][9]
    Rc, pc = camera_pose(scene, st, cam)
    D = pixel_directions(scene, cam, dx, dy) @ Rc.T
    npx = len(D)
    best, vis, piece, shade = np.full(npx, far), np.full(npx, -1), np.full(npx, -1), np.zeros(npx)
    t_err, n_err = np.zeros(npx), np.zeros(npx)
    T = np.full((nv, npx), np.inf) if keep_entries else None
    dist = np.zeros(nv)
    for s, (R, p) in enumerate(visual_poses(scene, st)):
        o, u = R.T @ (pc - p), D @ R
        dist[s] = np.linalg.norm(o)
        # only the rays that reach the bounding sphere can enter the shape (a cull of the reference's own; the result is the same)
        r = VF[s, 15] * (1 + 1e-9) + 1e-12
        b, c2 = u @ o, o @ o - r * r
        idx = np.nonzero((c2 <= 0) | ((b <= 0) & (b * b >= c2 * np.sum(u * u, axis=1))))[0]
        if not len(idx):
            continue
        t, nn, pcs, te, ne = entry(int(VI[s, 1]), VF[s, 7:11], o, u[idx])
        if keep_entries:
            T[s, idx] = t
        upd = (t >= near) & (t < best[idx])                          # in index order, strictly nearer: the first wins a tie
        k = idx[upd]
        best[k], vis[k], piece[k], t_err[k], n_err[k] = t[upd], s, pcs[upd], te[upd], ne[upd]
        shade[k] = 0.4 + 0.6 * np.maximum((nn[upd] @ R.T) @ LIGHT, 0.0)
    hit = vis >= 0
    colors = prm[h['P_COLOR']:h['P_COLOR'] + 3 * nv].reshape(nv, 3)
    rgb = np.where(hit[:, None], colors[np.maximum(vis, 0)] * shade[:, None] if nv else 1.0, 1.0)
    rgb_err = np.where(hit, 0.6 * colors[np.maximum(vis, 0)].max(axis=1) * n_err if nv else 0.0, 0.0)   # |d shade / d n| <= 0.6
    out = dict(vis=vis, t=best, rgb=rgb, piece=piece, near=near, far=far, t_err=t_err, rgb_err=rgb_err)
    if keep_entries:
        out.update(T=T, Tacc=np.where((T >= near) & (T < far), T, np.inf), dist=dist)
    return out


def render(scene, st, prm, cam):
    """fp64 image of camera `cam` for one environment: dict of rgb [H, W, 3], depth [H, W] (-t), seg [H, W] (body ids, -1
    background), `ambiguous` [H, W] and `allowed` [H, W, k] (mask values an fp32 renderer may show on ambiguous pixels, padded
    with the pixel's own value), and `ill_conditioned` [H, W]: the hit is certain but turning the ray by RAY_EPS would change its
    depth or colour by more than COND_DEPTH / COND_RGB (rays grazing a surface), so fp32 depth and colour may be off by more.

    A pixel is ambiguous where
      - the hit visual or its surface piece changes when the ray moves by JITTER pixels in x or y (silhouettes, edges, seams;
        the depth and colour of a hit change smoothly within a piece, so a fixed threshold on them would mark every slanted
        surface instead of the discontinuities);
      - some shape's entry lies within NEAR_TOL (relative to near, or far, plus the distance of the shape) of the near or the far
        plane: fp32 may accept what fp64 rejects and the other way round;
      - another shape's accepted entry lies within TIE_TOL (relative) of the hit, but not exactly on it: coincident surfaces
        computed from the same numbers tie exactly in both precisions and go to the lower index."""
    st, prm = np.asarray(st, np.float64), np.asarray(prm, np.float64)
    w, h = int(scene.sec['CAM_I'][cam][1]), int(scene.sec['CAM_I'][cam][2])
    VI = scene.sec['VIS_I']
    body = np.append(VI[:, 3].astype(float), -1.0)                  # body[-1] = background
    c = cast(scene, st, prm, cam, keep_entries=True)
    th = np.tan(scene.sec['CAM_F'][cam][7] * np.pi / 360.0)
    pix = (2 * th * w / h / w, 2 * th / h)                            # a pixel, in radians at the centre of the image
    near, far, T, Tacc, dist = c['near'], c['far'], c['T'], c['Tacc'], c['dist'][:, None]
    amb, ill = np.zeros(w * h, bool), np.zeros(w * h, bool)
    allowed = [body[c['vis']]]
    for dx, dy in ((JITTER, 0.0), (-JITTER, 0.0), (0.0, JITTER), (0.0, -JITTER)):
        j = cast(scene, st, prm, cam, dx, dy)
        amb |= (j['vis'] != c['vis']) | (j['piece'] != c['piece'])
        scale = JITTER * pix[0 if dx else 1] / RAY_EPS
        ill |= (np.abs(j['t'] - c['t']) > COND_DEPTH * scale * c['t']) | (np.abs(j['rgb'] - c['rgb']).max(axis=1) > COND_RGB * scale)
        allowed.append(body[j['vis']])
    with np.errstate(invalid='ignore'):
        plane = (np.abs(T - near) <= NEAR_TOL * (near + dist)) | (np.abs(T - far) <= NEAR_TOL * (far + dist))
        gap = np.abs(Tacc - c['t'][None, :])
        tie = (gap > 0) & (gap <= TIE_TOL * (c['t'][None, :] + dist))
    flagged = plane | tie
    amb |= flagged.any(axis=0)
    if len(VI):
        # an fp32 renderer may take any flagged shape, or, rejecting the hit at a plane, the shape behind it
        rest = Tacc.copy()
        rest[np.maximum(c['vis'], 0), np.arange(w * h)] = np.where(c['vis'] >= 0, np.inf, rest[0])
        second = np.where(rest.min(axis=0) < np.inf, np.argmin(rest, axis=0), -1)
        allowed.append(body[second])
        for s in np.unique(np.nonzero(flagged)[0]):
            allowed.append(np.where(flagged[s], body[s], body[c['vis']]))
    seg = body[c['vis']]
    return dict(rgb=c['rgb'].reshape(h, w, 3), depth=-c['t'].reshape(h, w), seg=seg.reshape(h, w), vis=c['vis'].reshape(h, w),
                depth_err=c['t_err'].reshape(h, w), rgb_err=c['rgb_err'].reshape(h, w),
                ambiguous=amb.reshape(h, w), ill_conditioned=(ill & ~amb).reshape(h, w), allowed=np.stack(allowed, axis=-1).reshape(h, w, -1))
