"""Timing of the ray_sensor add-on on the B200: dg_ray_kernel alone, and a full step of r2d2_maze with a 64-ray head lidar against
the same step without it (the two worlds alternated in one process).  Prints ms, rays/s and ray-shape tests/s (counted from the
scene's shapes), with the card's name and power limit read in the same run.

    python tools/ray_probe.py [--envs 4096] [--launches 200] [--steps 200] [--out DIR/ray_probe.json]

Also the home of `maze_with_lidar`, the lidar workload the tests use: r2d2_maze.yaml with a ray_sensor inserted under `r2d2`."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from diy_gym_b200.config import Configuration  # noqa: E402

MAZE = os.path.join(ROOT, 'examples', 'r2d2_maze', 'r2d2_maze.yaml')
LIDAR = dict(addon='ray_sensor', frame='head_swivel', xyz=[0, 0, 0], rpy=[0, 0, 0], range=[0.05, 8.0], num_rays=64,
             horizontal_fov=360, vertical_angles=[0])


def maze_with_lidar(with_lidar=True, **overrides):
    """The r2d2_maze configuration, with a head lidar on the R2D2 (keys of LIDAR, replaced by `overrides`).  The sensor sits at the
    centre of the head, 0.8 m above the ground: the maze's walls are 1 m tall."""
    with open(MAZE) as f:
        node = yaml.load(f, Loader=yaml.FullLoader)
    if with_lidar:
        node['r2d2']['lidar'] = dict(LIDAR, **overrides)
    return Configuration.from_dict('r2d2_maze_lidar' if with_lidar else 'r2d2_maze', node)


def ray_ops(scene):
    """(obs offset, rays, include_hit_object) of every ray_sensor op of a compiled scene."""
    from diy_gym_b200.compiler.scene import KERNEL_OPS
    return [(o['obs_off'], o['iargs'][1], bool(o['iargs'][2] & 1)) for o in scene.builder.ops if o['type'] == KERNEL_OPS['RAY_SENSOR']]


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--launches', type=int, default=200)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()

    import torch
    from diy_gym_b200.backend import World
    from diy_gym_b200.diy_gym import DIYGym

    if not torch.cuda.is_available():
        raise SystemExit('ray_probe: no CUDA device (there is no CPU measurement)')
    card = gpu_info()
    scenes = {k: DIYGym(maze_with_lidar(k == 'lidar'), num_envs=1, compile_only=True).scene for k in ('lidar', 'plain')}
    worlds = {k: World(sc, args.envs, seed=7) for k, sc in scenes.items()}
    for w in worlds.values():
        w.reset()
        w.action.uniform_(-0.5, 0.5)
        for _ in range(20):   # warm-up: modules loaded, the adaptive schedule settled
            w.step()
    torch.cuda.synchronize()

    sc = scenes['lidar']
    rays = sum(r for _, r, _ in ray_ops(sc))
    ns = sc.hdr['ns']
    n_static = int(sum(sc.sec['SHAPE_I'][:, 3] != 0))
    tests = args.envs * rays * ns   # bounding-sphere tests: every ray against every collision shape

    # dg_ray_kernel alone, two ways: (1) CUDA events around `launches` observe() calls of the lidar world ([step kernel in observe
    # mode, dg_ray_kernel]) minus the same for the world without the lidar (the first launch only); (2) the kernel's own durations
    # from torch.profiler in a separate pass.
    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    res = {'card': card, 'envs': args.envs, 'rays_per_env': rays, 'shapes': ns, 'static_shapes': n_static,
           'observe_ms': {'lidar': [], 'plain': []}, 'step_ms': {'lidar': [], 'plain': []}}
    for _ in range(args.rounds):
        for k in ('lidar', 'plain'):
            w = worlds[k]
            timed(w.observe, 10)
            res['observe_ms'][k].append(timed(w.observe, args.launches))
        for k in ('lidar', 'plain'):
            w = worlds[k]
            res['step_ms'][k].append(timed(w.step, args.steps))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.launches):
            worlds['lidar'].observe()
        torch.cuda.synchronize()
    durs = [e.device_time for e in prof.events() if 'dg_ray_kernel' in e.name]   # microseconds
    res['ray_kernel_profiler_ms'] = float(np.median(durs)) * 1e-3 if durs else None
    res['ray_kernel_profiler_launches'] = len(durs)
    med = lambda v: float(np.median(v))
    ray_ms = med(res['observe_ms']['lidar']) - med(res['observe_ms']['plain'])
    res['ray_kernel_ms'] = ray_ms
    res['rays_per_s'] = args.envs * rays / (ray_ms * 1e-3) if ray_ms > 0 else None
    res['ray_shape_tests_per_s'] = tests / (ray_ms * 1e-3) if ray_ms > 0 else None
    res['step_ms_median'] = {k: med(v) for k, v in res['step_ms'].items()}
    print(json.dumps(res))
    print('%s | %d envs x %d rays x %d shapes (%d static): dg_ray_kernel %.4f ms by events, %s ms by the profiler '
          '(%.3g rays/s, %.3g ray-shape tests/s); step with lidar %.4f ms, without %.4f ms'
          % (card, args.envs, rays, ns, n_static, ray_ms, res['ray_kernel_profiler_ms'], res['rays_per_s'] or 0,
             res['ray_shape_tests_per_s'] or 0, res['step_ms_median']['lidar'], res['step_ms_median']['plain']))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)
    for w in worlds.values():
        w.close()


if __name__ == '__main__':
    main()
