"""Timing of the dynamics queries on the B200 (Model.jacobian / mass_matrix / inverse_dynamics, and one dg_body_dynamics call that
computes all three outputs), for the UR5 of ur_high_5 at 1024 and 8192 environments and for the Jaco (10 DoF) and the floating
R2D2 (n = 14) of from_the_readme at 4096.  Each number is the median over `--rounds` alternated rounds of CUDA events around
`--calls` calls after a warm-up; a step of the same world is timed the same way for scale.  The card's name and power limit are
read in the same run.

    python tools/dynamics_probe.py [--calls 200] [--rounds 5] [--out DIR/dynamics_probe.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [('ur_high_5', 'ur5_l', 1024), ('ur_high_5', 'ur5_l', 8192), ('from_the_readme', 'robot', 4096), ('from_the_readme', 'r2d2', 4096)]


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

    if not torch.cuda.is_available():
        raise SystemExit('dynamics_probe: no CUDA device (there is no CPU measurement)')
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
    for name, model, n_envs in CASES:
        env = DIYGym(os.path.join(ROOT, 'examples', name, name + '.yaml'), num_envs=n_envs, device=0, seed=7)
        g = torch.Generator(device='cuda').manual_seed(0)
        for _ in range(10):
            env.step(env.sample_action(g))
        m, w = env.models[model], env.world
        n = m.body.n_dofs + (6 if m.body.kind == 2 else 0)
        link = m.num_joints() - 1
        qdd = torch.rand((n_envs, n), device='cuda')
        fns = {'jacobian': lambda: m.jacobian(link, (0., 0., 0.05)),
               'mass_matrix': lambda: m.mass_matrix(),
               'inverse_dynamics': lambda: m.inverse_dynamics(qdd=qdd),
               'body_dynamics_all': lambda: w.body_dynamics(m.uid, link, (0., 0., 0.05), None, None, qdd, jac=True, mass=True, tau=True),
               'step': w.step}
        for f in fns.values():   # warm-up: modules loaded, allocator primed
            timed(f, 20)
        ms = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, f in fns.items():
                ms[k].append(timed(f, args.calls))
        rec = {'config': name, 'model': model, 'n': n, 'envs': n_envs, 'ms_median': {k: float(np.median(v)) for k, v in ms.items()},
               'ms_rounds': ms, 'output_floats_per_env': 6 * n + n * n + n}
        results.append(rec)
        print('%s %s n=%d %d envs: %s' % (name, model, n, n_envs, ', '.join('%s %.4f ms' % kv for kv in rec['ms_median'].items())))
        env.close()
    res = {'card': card, 'calls_per_round': args.calls, 'rounds': args.rounds, 'results': results}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
