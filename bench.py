#!/usr/bin/env python
"""bench.py - throughput of the DIYGym step path on B200(s): aggregate env-steps/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--envs E] [--impl ours|reference] [--dump-outputs DIR]

One step = one DIYGym.step for every environment (add-on update -> 2 x 1/480 s physics sub-steps with 150 solver
sweeps -> observe/reward/terminal), synthetic uniform random actions.  Default workload = BASELINE.json configs[1]:
examples/r2d2_maze (maze_size 10, 119 walls), 4096 environments per GPU.  Other configs: --config ur_high_5
(8192/GPU), from_the_readme (4096/GPU, 200x200 camera every step), drone_pilot (4096/GPU), ur_high_5_randomised.

Printed JSON line (rank 0):
  value      whole-job env-steps/s, actions already resident in HBM, CUDA-event timed, max over ranks
  e2e        the same through the host-buffer C-ABI call dg_step_host (pinned host actions H2D, outputs D2H, per step)
  roofline   dominant kernel dg_step_kernel against the measured HBM peak (algorithmic bytes per env-step from
             DESIGN.md) plus, under "fp32", its oracle-counted flops against the measured FMA peak - the bound that
             actually binds the physics-only configs
  cpu_baseline  the CPU oracle (kind "port", this repo's fp64 restatement - pybullet is absent) on the host cores
With --impl reference the oracle itself is the timed arm (all host threads, bounded sample).
Under torchrun (--gpus N > 1) every rank owns its own N environments (no per-step collective, weak scaling).

--dump-outputs DIR writes what the last timed step left in rank 0's device buffers, as float32 DIR/<name>.npy: `state`
(the physics state rows), `obs`, `reward`, `term` (the zero-width ones of a config are skipped) and `camera<k>_rgb` /
`camera<k>_depth` per camera.  In configs with terminals, the step ends with the masked reset of finished episodes, and
`reset` is 1 for the environments it restarted.  The reset observes them again, so in their rows `state`, `obs`,
`reward` and `term` are post-reset values; the images are rendered before the reset.  Above 64 MB in all, a fixed sample of environments (seeded, the same rows in every
array) is written instead; `env_index.npy` (float64) lists the environments written.  Actions, seeds and the step
sequence depend only on the arguments, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (yaml path, envs per GPU, action scale)
    'r2d2_maze': ('examples/r2d2_maze/r2d2_maze.yaml', 4096),
    'ur_high_5': ('examples/ur_high_5/ur_high_5.yaml', 8192),
    'ur_high_5_randomised': ('examples/ur_high_5/ur_high_5_randomised.yaml', 8192),
    'from_the_readme': ('examples/from_the_readme/from_the_readme.yaml', 4096),
    'drone_pilot': ('examples/drone_pilot/drone_pilot.yaml', 4096),
    'basic_env': ('examples/basic_env/basic_env.yaml', 4096),
    'ur_admittance': ('examples/ur_admittance/ur_admittance.yaml', 8192),
    'ur_gripper': ('examples/ur_gripper/ur_gripper.yaml', 4096),
    'ur_extras': ('examples/ur_extras/ur_extras.yaml', 4096),
    'ur_robotiq': ('examples/ur_gripper/ur_robotiq.yaml', 4096),
}
METRIC = 'aggregate env-steps/sec'
UNIT = 'env-steps/s'


def action_ranges(env):
    """(low, high) rows of the flattened device action buffer, from the add-on action spaces; the maze wheels get the
    example's +-10 rad/s instead of the +-0.5 of the space (SURVEY 8d)."""
    import numpy as np
    n_act = env.scene['n_act']
    lo, hi = np.zeros(n_act, np.float32), np.zeros(n_act, np.float32)
    for op in env.builder.ops:
        if op['n_act']:
            lo[op['act_off']:op['act_off'] + op['n_act']] = -1.0
            hi[op['act_off']:op['act_off'] + op['n_act']] = 1.0
    for r in env.receptors.values():
        for a in r.addons.values():
            op = getattr(a, 'op', None)
            if op is None or not op['n_act']:
                continue
            from diy_gym_b200.utils import flatten, get_bounds_for_space
            l = np.asarray(flatten(get_bounds_for_space(a.action_space, True), batched=False), np.float32).reshape(-1)
            h = np.asarray(flatten(get_bounds_for_space(a.action_space, False), batched=False), np.float32).reshape(-1)
            if type(a).__name__ == 'JointController' and env.name == 'r2d2_maze':
                l, h = l * 20.0, h * 20.0
            lo[op['act_off']:op['act_off'] + op['n_act']] = l
            hi[op['act_off']:op['act_off'] + op['n_act']] = h
    return lo, hi


def register_example_addons():
    import importlib.util
    spec = importlib.util.spec_from_file_location('drone_pilot_example', os.path.join(ROOT, 'examples', 'drone_pilot', 'drone_pilot.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, device):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(device), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 8 and r[0].replace('.', '').isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace('.', '').isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 8:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons), 'samples': len(sm)}


def cpu_oracle_rate(scene, lo, hi, seconds=12.0, threads=None, seed=1234):
    """env-steps/s of the fp64 CPU oracle (oracle/bullet_restatement.c, one world per environment, pthreads over
    environments) on a bounded sample of the workload."""
    import ctypes
    import numpy as np
    from oracle import oracle as orc
    L = orc.lib()
    threads = threads or L.dgo_batch_max_threads()
    n_env = max(threads * 2, 8)
    worlds = [orc.OracleWorld(scene, seed=seed, env_id=i) for i in range(n_env)]
    arr = (ctypes.c_void_p * n_env)(*[w._w for w in worlds])
    L.dgo_batch_reset(arr, n_env, threads)
    h = scene.hdr
    rng = np.random.default_rng(seed)
    obs = np.zeros((n_env, max(h['n_obs'], 1)))
    rew = np.zeros((n_env, max(h['n_rew'], 1)))
    term = np.zeros((n_env, max(h['n_term'], 1)), np.uint8)
    dp = ctypes.POINTER(ctypes.c_double)

    def run(nsteps):
        act = rng.uniform(lo, hi, (nsteps, n_env, h['n_act'])) if h['n_act'] else np.zeros((nsteps, n_env, 1))
        t0 = time.perf_counter()
        L.dgo_batch_step(arr, n_env, nsteps, act.ctypes.data_as(dp), h['n_act'], obs.ctypes.data_as(dp), h['n_obs'], rew.ctypes.data_as(dp),
                         h['n_rew'], term.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), h['n_term'], threads)
        return time.perf_counter() - t0
    run(2)
    # flop counter of the oracle (SURVEY 8d "algorithmic work"): single-threaded probe, the counter is not atomic
    probe = orc.OracleWorld(scene, seed=seed, env_id=0)
    probe.env_reset()
    orc.flops(reset=True)
    for _ in range(4):
        probe.env_step(rng.uniform(lo, hi) if h['n_act'] else np.zeros(1))
    flops_per_step = orc.flops(reset=True) / 4.0
    t_probe = run(4)
    nsteps = int(max(4, min(2000, seconds / max(t_probe / 4, 1e-6))))
    dt = run(nsteps)
    return {'value': n_env * nsteps / dt, 'unit': UNIT, 'cores': int(threads), 'kind': 'port',
            'sample': '%d envs x %d steps of %s on %d threads (fp64 oracle; pybullet is not installed)' % (n_env, nsteps, h.get('name', 'the workload'), threads),
            'flops_per_env_step': flops_per_step}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--config', default='r2d2_maze', choices=sorted(CONFIGS))
    ap.add_argument('--envs', type=int, default=0, help='environments per GPU (default: the config\'s BASELINE.json size)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--team', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-per-config', action='store_true', help='skip the short runs of the other BASELINE.json configs (default run, 1 GPU)')
    ap.add_argument('--preroll', type=int, default=300, help='untimed steps before the warm-up (contact counts stationarise)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the CUDA step path (--impl ours)')

    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world_size = int(os.environ.get('WORLD_SIZE', 1))
    path, envs_default = CONFIGS[args.config]
    n_envs = args.envs or envs_default
    warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    register_example_addons()
    from diy_gym_b200 import DIYGym
    from diy_gym_b200.config import Configuration

    cfg_workload = {'workload': '%s, %d envs/GPU, 2 sub-steps x 150 solver sweeps at 1/240 s, uniform random actions' % (args.config, n_envs),
                    'envs_per_gpu': n_envs, 'parallelism': 'env-sharded x%d, no per-step collective' % max(args.gpus, 1)}

    # ---------------------------------------------------------------- reference arm: the CPU oracle ----------------
    if args.impl == 'reference':
        if rank != 0:
            return 0
        env = DIYGym(Configuration.from_file(os.path.join(ROOT, path)), num_envs=1, compile_only=True)   # host-side scene compile only
        lo, hi = action_ranges(env)
        vals, base = [], None
        for _ in range(warmup and 1):
            cpu_oracle_rate(env.scene, lo, hi, seconds=1.0)
        per = min(8.0, 120.0 / args.steps)   # --steps timed samples of about 120 s in all
        for _ in range(args.steps):
            base = cpu_oracle_rate(env.scene, lo, hi, seconds=per)
            vals.append(base['value'])
        v = float(np.median(vals))
        base['value'] = v
        line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': warmup,
                'ms_per_step': None, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': cfg_workload, 'cpu_baseline': base,
                'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- our arm ----------------------------------------
    if world_size > 1:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    ctx = dict(rank=rank, local_rank=local_rank, world_size=world_size, dev=dev, warmup=warmup, steps=args.steps, preroll=args.preroll, team=args.team)
    main_res = measure(args.config, n_envs, ctx, cpu_baseline=not args.no_cpu_baseline, api_leg=True, dump_dir=args.dump_outputs)
    # the other BASELINE.json configs, one GPU only: the same measurement with the same number of timed steps, shorter pre-roll
    per_config = None
    if world_size == 1 and not args.no_per_config and args.config == 'r2d2_maze' and not args.envs:
        per_config = {}
        for name in ('ur_high_5', 'from_the_readme', 'drone_pilot', 'ur_high_5_randomised'):
            r = measure(name, CONFIGS[name][1], dict(ctx, preroll=min(args.preroll, 200)), cpu_baseline=False, api_leg=False)
            per_config['%s@%d' % (name, CONFIGS[name][1])] = {k: r[k] for k in ('value', 'ms_per_step', 'kernel_ms', 'e2e', 'roofline', 'gpu_launches', 'split_schedule')}
    if rank != 0:
        if world_size > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return 0
    r = main_res
    line = {'metric': METRIC, 'value': r['value'], 'unit': UNIT, 'n_gpus': world_size, 'steps': args.steps, 'warmup': warmup,
            'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': dict(cfg_workload, **r['config_extra']), 'e2e': r['e2e'], 'e2e_api': r.get('e2e_api'),
            'gpu_launches': r['gpu_launches'], 'clocks': r['clocks'], 'roofline': r['roofline'], 'cpu_baseline': r['cpu_baseline']}
    if per_config is not None:
        line['per_config'] = per_config
    print(json.dumps(line))
    if world_size > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


def measure(config, n_envs, ctx, cpu_baseline=True, api_leg=True, dump_dir=None):
    """One configuration on this rank's GPU: pre-roll, K timed steps (device-resident actions, CUDA events, L2 flushed before
    every timed step), the host-buffer leg through dg_step_host, optionally the same loop through DIYGym.step(action dict), the
    roofline of the step launch sequence and the CPU oracle beside it.  Every rank calls this with the same arguments (the
    barriers and the max-over-ranks reduction are inside).  dump_dir: rank 0 writes the outputs of the last timed step there."""
    import numpy as np
    import torch
    from diy_gym_b200 import DIYGym
    rank, local_rank, world_size, dev = ctx['rank'], ctx['local_rank'], ctx['world_size'], ctx['dev']
    warmup, steps = ctx['warmup'], ctx['steps']
    path = CONFIGS[config][0]
    env = DIYGym(os.path.join(ROOT, path), num_envs=n_envs, device=local_rank, seed=1234, team=ctx['team'], env_id_offset=rank * n_envs)
    w, sc = env.world, env.scene
    lo_np, hi_np = action_ranges(env)
    lo, hi = torch.from_numpy(lo_np).to(dev), torch.from_numpy(hi_np).to(dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    n_pool = 8   # pre-generated action batches, resident in HBM, cycled (different actions every step)
    pool = [lo + (hi - lo) * torch.rand((n_envs, w.n_act), device=dev, generator=g) for _ in range(n_pool)] if w.n_act else None
    user_addons = [a for r in env.receptors.values() for a in r.addons.values() if getattr(a, 'op', None) is None and a.action_space is not None]
    cams = [a for r in env.receptors.values() for a in r.addons.values() if type(a).__name__ == 'Camera']
    has_term = w.n_term > 0
    last = {}   # the last step's images (views of buffers the next render overwrites) and reset mask, for --dump-outputs

    def device_step(i, render=True):
        if pool is not None:
            w.action.copy_(pool[i % n_pool])
        for a in user_addons:   # user add-ons that stayed in Python run their batched torch update
            a.update(torch.rand((n_envs, ) + tuple(a.action_space.shape), device=dev, generator=g))
        w.step()
        if render:
            for k, c in enumerate(cams):
                last['camera%d_rgb' % k], last['camera%d_depth' % k] = w.render(c.cam)
        if has_term:
            last['reset'] = w.term.amax(dim=1)
            w.reset(last['reset'])   # masked reset of finished episodes, no host sync

    def barrier():
        if world_size > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    # Pre-roll (untimed): the first steps after a reset are not representative - the robots are still falling onto their
    # wheels / the table, contact counts and with them the solver work grow for ~100 steps - so the timed window starts after
    # `preroll` steps, when --steps 20 and --steps 1000 read the same.  Cameras are not rendered during the pre-roll.
    for i in range(ctx['preroll']):
        device_step(i, render=False)
    # L2 flush between timed iterations: a buffer twice the size of the 126 MB L2 is overwritten before every timed
    # step (outside the per-step CUDA-event brackets), so that every step starts with state, parameters and actions
    # in HBM, not in L2
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for i in range(warmup):
        device_step(i)
    barrier()
    l0 = w.launches
    sampler = ClockSampler(local_rank) if rank == 0 else None
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    step_plain = w.step

    def step_timed(i):
        kev[i][0].record()
        step_plain()
        kev[i][1].record()
    sev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush_buf.fill_(float(i))               # L2 flush (a torch fill kernel: not counted in gpu_launches, not timed)
        w.step = lambda i=i: step_timed(i)      # CUDA events around the step's launch sequence, on the launching stream
        sev[i][0].record()
        device_step(warmup + i)
        sev[i][1].record()
    w.step = step_plain
    barrier()
    ms_total = float(sum(a.elapsed_time(b) for a, b in sev))   # the K timed steps, device time, flushes excluded
    launches = w.launches - l0
    clocks = sampler.stop() if sampler else None
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))   # average duration of a step's launches inside the timed region
    if dump_dir and rank == 0:   # before the legs below step the world further
        dump_outputs(dump_dir, dict(state=w.state, obs=w.obs, reward=w.reward, term=w.term, **last), n_envs)

    # ---- end to end through the host-buffer C-ABI call ----------------------------------------------------------
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
    act_h = pin((n_envs, max(w.n_act, 1)), torch.float32)[:, :w.n_act]
    obs_h, rew_h, term_h = pin((n_envs, max(w.n_obs, 1)), torch.float32), pin((n_envs, max(w.n_rew, 1)), torch.float32), pin((n_envs, max(w.n_term, 1)), torch.uint8)
    extra_h = torch.empty((n_envs, 13), dtype=torch.float32).pin_memory()
    rng = np.random.default_rng(99 + rank)
    host_pool = [(lo_np + (hi_np - lo_np) * rng.random((n_envs, w.n_act), dtype=np.float32)) for _ in range(4)] if w.n_act else None
    cam_h = [tuple(torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in w.render(c.cam)) for c in cams]
    cam_h8 = [tuple(torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in w.render(c.cam, u8=True)) for c in cams]   # colour as bytes (dg_render_u8)
    h2d = n_envs * w.n_act * 4
    d2h = n_envs * (w.n_obs * 4 + w.n_rew * 4 + w.n_term)
    dyn_body = next((b for b in sc.bodies if b.kind != 0), sc.bodies[0])
    o_pose = sc.hdr['S_BPOS'] + 3 * dyn_body.index
    if d2h == 0:
        d2h = n_envs * 3 * 4   # no sensor in this config: read back the robot's base position as the step's result
    d2h_u8 = d2h + sum(int(t.numel() * t.element_size()) for pair in cam_h8 for t in pair)
    d2h += sum(int(t.numel() * t.element_size()) for pair in cam_h for t in pair)

    def host_step(i, u8=False):
        if host_pool is not None:
            np.copyto(act_h, host_pool[i % 4])
        for a in user_addons:
            a.update(torch.rand((n_envs, ) + tuple(a.action_space.shape), device=dev, generator=g))
        w.step_host(act_h if w.n_act else None, obs_h if w.n_obs else None, rew_h if w.n_rew else None, term_h if w.n_term else None)
        if w.n_obs + w.n_rew + w.n_term == 0:
            extra_h[:, :3].copy_(w.state[:, o_pose:o_pose + 3])
        for c, hs in zip(cams, cam_h8 if u8 else cam_h):
            for t_h, t_d in zip(hs, w.render(c.cam, u8=u8)):
                t_h.copy_(t_d, non_blocking=True)
        if cams:
            torch.cuda.synchronize(dev)
        if has_term and term_h[:, :w.n_term].any():
            w.reset(torch.from_numpy(term_h[:, :w.n_term].max(axis=1)))
    for i in range(3):
        host_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        host_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_u8_s = 0.0
    if cams:   # the same with the colour images as bytes (camera key `rgb_uint8`, dg_render_u8): what a host-side consumer would ask for
        for i in range(2):
            host_step(i, u8=True)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            host_step(i, u8=True)
        barrier()
        e2e_u8_s = time.perf_counter() - t0

    # ---- the same through the public Python API: DIYGym.step(action dict) -> (obs, reward, terminal) dicts, consumed ---------
    api_s, api_bytes = 0.0, (0, 0)
    if api_leg:
        from diy_gym_b200 import spaces as dg_spaces
        leaves = []   # (path, pinned host tensor) per action leaf, in action_space order

        def collect(sp, pth):
            if isinstance(sp, dg_spaces.Dict):
                for k, v in sp.spaces.items():
                    collect(v, pth + (k, ))
            else:
                lo_l, hi_l = np.asarray(sp.low, np.float32), np.asarray(sp.high, np.float32)
                if config == 'r2d2_maze':
                    lo_l, hi_l = lo_l * 20.0, hi_l * 20.0
                leaves.append((pth, torch.empty((n_envs, ) + tuple(sp.shape), dtype=torch.float32).pin_memory(), lo_l, hi_l))
        collect(env.action_space, ())
        out_h = {}

        def consume(tree, pth=()):
            """device -> pinned host copy of every leaf of a returned tree (the bytes a learner on the host would read)"""
            n = 0
            if isinstance(tree, dict):
                for k, v in tree.items():
                    n += consume(v, pth + (k, ))
            elif isinstance(tree, torch.Tensor):
                if pth not in out_h:
                    out_h[pth] = torch.empty(tree.shape, dtype=tree.dtype).pin_memory()
                out_h[pth].copy_(tree, non_blocking=True)
                n += tree.numel() * tree.element_size()
            return n

        def api_step(i):
            action, nb_in = {}, 0
            for pth, t_h, lo_l, hi_l in leaves:
                t_h.copy_(torch.from_numpy(lo_l + (hi_l - lo_l) * rng.random(t_h.shape, dtype=np.float32)))
                d = action
                for k in pth[:-1]:
                    d = d.setdefault(k, {})
                d[pth[-1]] = t_h.to(dev, non_blocking=True)
                nb_in += t_h.numel() * 4
            obs, rew, term, _ = env.step(action)
            nb_out = consume(obs, ('obs', )) + consume(rew, ('rew', )) + consume(term, ('term', ))
            torch.cuda.synchronize(dev)
            done = out_h.get(('term', ))
            if has_term:
                flat = [v for k, v in out_h.items() if k[0] == 'term']
                if any(bool(v.any()) for v in flat):
                    w.reset(w.term.amax(dim=1))
            return nb_in, nb_out
        for i in range(3):
            api_bytes = api_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            api_step(i)
        barrier()
        api_s = time.perf_counter() - t0

    # ---- max over ranks --------------------------------------------------------------------------------------------
    stats = torch.tensor([ms_total, e2e_s, kernel_ms, api_s, e2e_u8_s], dtype=torch.float64, device=dev)
    if world_size > 1:
        import torch.distributed as dist
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_total, e2e_s, kernel_ms, api_s, e2e_u8_s = [float(x) for x in stats.tolist()]
    res = {'config_extra': dict(team=w.team, block_threads=w.block_threads, grid_blocks=w.grid_blocks, smem_bytes=w.smem_bytes, split_schedule=bool(getattr(w, 'split', False)),
                                preroll_steps=ctx['preroll'], l2_policy='L2 flushed (256 MB buffer overwritten) before every timed step; per-step actions cycle through 8 pre-generated batches'),
           'split_schedule': bool(getattr(w, 'split', False))}
    if rank != 0:
        env.close()
        return res
    total_envs = n_envs * world_size
    res.update(value=total_envs * steps / (ms_total * 1e-3), ms_per_step=ms_total / steps, kernel_ms=kernel_ms, gpu_launches=int(launches), clocks=clocks,
               e2e={'value': total_envs * steps / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'api': 'dg_step_host (pinned host buffers)' + (' + dg_render, images D2H' if cams else '')})
    if cams:
        res['e2e']['rgb_uint8'] = {'value': total_envs * steps / e2e_u8_s, 'unit': UNIT, 'd2h_bytes_per_step': d2h_u8, 'api': 'dg_step_host + dg_render_u8 (colour as bytes, depth fp32), images D2H'}
    if api_leg:
        res['e2e_api'] = {'value': total_envs * steps / api_s, 'unit': UNIT, 'h2d_bytes_per_step': int(api_bytes[0]), 'd2h_bytes_per_step': int(api_bytes[1]),
                          'api': 'DIYGym.step(action dict): pinned host actions H2D, every leaf of the returned obs / reward / terminal trees D2H'}

    # ---- roofline of the step's launch sequence ------------------------------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    # algorithmic bytes per env-step (DESIGN.md "bytes per unit"): dynamic state read + written, action, outputs
    dyn_state = sum(13 for b in sc.bodies if b.kind != 0) + 9 * sc['nd'] + 13 * sc['nl'] + 2
    alg_bytes = 4 * (2 * dyn_state + w.n_act + w.n_obs + w.n_rew) + w.n_term
    img_bytes = sum(int(t.numel() * t.element_size()) for c in cams for t in w.render(c.cam)) // n_envs
    from diy_gym_b200.backend import measure_fp32_peak
    fp32_peak = measure_fp32_peak(local_rank)
    cpu = cpu_oracle_rate(sc, lo_np, hi_np) if cpu_baseline else None
    flops = cpu['flops_per_env_step'] if cpu else oracle_flops(sc, lo_np, hi_np)
    traffic = render_traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of one step's launches / of one render launch (ncu, profiles/ncu_traffic.json)
    try:
        table = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
        traffic, render_traffic = table.get('%s:%d' % (config, n_envs)), table.get('%s:%d:render' % (config, n_envs))
    except Exception:
        pass
    kname = ('dg_step_kernel<%d> stage launches + dg_solve_kernel' % w.team) if res['split_schedule'] else 'dg_step_kernel<%d>' % w.team
    hbm = {'achieved': alg_bytes * n_envs / (kernel_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s', 'algorithmic_bytes_per_env_step': alg_bytes,
           'peak_source': 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback'}
    hbm['frac'] = hbm['achieved'] / hbm_peak
    tf = flops * n_envs / (kernel_ms * 1e-3) / 1e12
    fp32 = {'achieved': tf, 'peak': fp32_peak, 'unit': 'TFLOP/s', 'frac': tf / fp32_peak if fp32_peak else None, 'flops_per_env_step': flops,
            'peak_source': 'measured FMA micro-kernel (dg_measure_fp32_peak)'}
    # the binding bound goes on top: non-tensor FP32 issue for the physics, HBM writes for a config that renders images every step
    if cams:
        render_ms = max(ms_total / steps - kernel_ms, 1e-6)
        a = img_bytes * n_envs / (render_ms * 1e-3) / 1e9
        roofline = {'bound': 'hbm', 'kernel': 'dg_render_kernel', 'achieved': a, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': a / hbm_peak, 'traffic': render_traffic,
                    'peak_source': hbm['peak_source'], 'algorithmic_bytes_per_env_step': img_bytes, 'kernel_ms': render_ms,
                    'note': 'the render launch (image bytes written per env-step) is the dominant kernel of this config; the physics launches are under "step"',
                    'step': dict(fp32, bound='fp32', kernel=kname, kernel_ms=kernel_ms, traffic=traffic, hbm=hbm)}
    else:
        roofline = dict(fp32, bound='fp32', kernel=kname, kernel_ms=kernel_ms, traffic=traffic,
                        note='bound = non-tensor FP32 issue (oracle-counted flops / measured FMA peak): the physics is a chain of small dependent fp32 systems; the HBM bound (algorithmic state bytes / measured copy bandwidth) is three orders of magnitude away and listed under "hbm"',
                        hbm=hbm)
    res.update(roofline=roofline, cpu_baseline=cpu)
    env.close()
    return res


DUMP_LIMIT = 64 * 1000 * 1000   # bytes


def dump_outputs(out_dir, arrays, n_envs):
    """Writes each [n_envs, ...] device tensor of `arrays` as float32 out_dir/<name>.npy, zero-width ones skipped.  Above
    DUMP_LIMIT bytes in all, the same seeded sample of environment rows is taken from every array."""
    import numpy as np
    import torch
    arrays = {k: v for k, v in arrays.items() if v.numel()}
    row_bytes = sum(4 * v[0].numel() for v in arrays.values()) + 8   # + the env_index entry
    keep = min(n_envs, (DUMP_LIMIT - 128 * (len(arrays) + 1)) // row_bytes)   # 128: the header of a .npy file
    idx = np.arange(n_envs) if keep == n_envs else np.sort(np.random.default_rng(0).choice(n_envs, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'env_index.npy'), idx.astype(np.float64))
    rows = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), v.index_select(0, rows).float().cpu().numpy())


def oracle_flops(scene, lo, hi, seed=1234):
    """flops per env-step from the oracle's instrumented counter (4 steps of one environment, single thread)"""
    import numpy as np
    from oracle import oracle as orc
    rng = np.random.default_rng(seed)
    probe = orc.OracleWorld(scene, seed=seed, env_id=0)
    probe.env_reset()
    for _ in range(30):
        probe.env_step(rng.uniform(lo, hi) if scene.hdr['n_act'] else np.zeros(1))
    orc.flops(reset=True)
    for _ in range(4):
        probe.env_step(rng.uniform(lo, hi) if scene.hdr['n_act'] else np.zeros(1))
    return orc.flops(reset=True) / 4.0


if __name__ == '__main__':
    sys.exit(main())
