"""Timing of the inverse-kinematics query on the B200 (Model.inverse_kinematics, one dg_ik_kernel launch per call): the UR5 of
ur_high_5 (pose target, null-space lists) at 1024 and 8192 environments, and the Jaco (position target, 10 DoF) and the floating
R2D2 (pose target, 8 DoF) of from_the_readme at 4096.  Targets are the link frame's current pose moved by 2 cm and rotated by
0.05 rad.  'ik' solves with the scene's defaults (20 iterations, early exit at 1e-4 m); 'ik_all_iterations' with threshold 0,
so that every lane runs all 20.  Each number is the median over `--rounds` alternated rounds of CUDA events around `--calls`
calls after a warm-up; a step of the same world is timed the same way for scale.  The card's name and power limit are read in
the same run.

    python tools/ik_probe.py [--calls 200] [--rounds 5] [--out DIR/ik_probe.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (config, model, link joint, orientation target, null-space lists, environments)
CASES = [('ur_high_5', 'ur5_l', 'ee_fixed_joint', True, True, 1024), ('ur_high_5', 'ur5_l', 'ee_fixed_joint', True, True, 8192),
         ('from_the_readme', 'robot', 'j2s7s300_joint_end_effector', False, False, 4096),
         ('from_the_readme', 'r2d2', 'left_tip_joint', True, False, 4096)]
REST = {'ur5_l': [-0.17, -0.73, -1.93, -0.36, -0.03, -0.06]}


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()

    import torch
    from diy_gym_b200 import DIYGym
    from diy_gym_b200 import torch_math as tm

    if not torch.cuda.is_available():
        raise SystemExit('ik_probe: no CUDA device (there is no CPU measurement)')
    card = gpu_info()

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    results = []
    for name, model, joint, use_orn, nullspace, n_envs in CASES:
        env = DIYGym(os.path.join(ROOT, 'examples', name, name + '.yaml'), num_envs=n_envs, device=0, seed=7)
        g = torch.Generator(device='cuda').manual_seed(0)
        for _ in range(10):
            env.step(env.sample_action(g))
        m, w = env.models[model], env.world
        link = m.get_frame_id(joint)
        pos, quat = m.get_transform(link)
        tpos = (pos + torch.tensor([0.02, -0.02, 0.02], device='cuda')).contiguous()
        torn = tm.quat_mul(quat, tm.quat_from_euler(torch.full_like(pos, 0.05))).contiguous() if use_orn else None
        kw = {}
        if nullspace:
            infos = [m.joint_info(i) for i in m.body.movable_joints()]
            lo, up = [i['lower'] for i in infos], [i['upper'] for i in infos]
            lists = (lo, up, [u - l for l, u in zip(lo, up)], REST[model])
            kw = dict(zip(('lower_limits', 'upper_limits', 'joint_ranges', 'rest_poses'), [torch.tensor(v, dtype=torch.float32, device='cuda') for v in lists]))
        fns = {'ik': lambda: m.inverse_kinematics(link, tpos, torn, **kw),
               'ik_all_iterations': lambda: m.inverse_kinematics(link, tpos, torn, residual_threshold=0.0, **kw),
               'step': w.step}
        for f in fns.values():   # warm-up: modules loaded, allocator primed, the world's IK buffer allocated
            timed(f, 20)
        ms = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, f in fns.items():
                ms[k].append(timed(f, args.calls))
        _, err = m.inverse_kinematics(link, tpos, torn, return_error=True, **kw)
        rec = {'config': name, 'model': model, 'link': joint, 'n_dof': m.body.n_dofs, 'orientation': use_orn, 'nullspace': nullspace,
               'envs': n_envs, 'ms_median': {k: float(np.median(v)) for k, v in ms.items()}, 'ms_rounds': ms,
               'err_median_m_rad': [float(x) for x in err.median(dim=0).values.cpu()]}
        results.append(rec)
        print('%s %s %d DoF %d envs: %s' % (name, model, m.body.n_dofs, n_envs, ', '.join('%s %.4f ms' % kv for kv in rec['ms_median'].items())))
        env.close()
    res = {'card': card, 'calls_per_round': args.calls, 'rounds': args.rounds, 'results': results}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
