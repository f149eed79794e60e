"""Cost of per-environment episodes (BatchedPhysics.reset_envs): the restart itself and the episode
clock on the step kernels.

  1. Device time of one fb_reset_envs_where (CUDA events on the engine's stream) at 65,536 swimming
     SALAMANDERs with 1 environment, 1 %, 10 % and 100 % of them masked, next to the host time of
     one fb_reset of the whole batch (it uploads every row and synchronises).
  2. Step throughput with the episode clock bound (an environment restarted after iteration 0:
     the ENVP = 1 kernels run) against unbound (no restart: the ENVP = 0 kernels), alternated round
     after round: 65,536 swimming SALAMANDERs (bench.py's headline configuration) and 4,096 on the
     ground.
  3. With --parent TREE (a checkout of the parent commit, built): bench.py's headline line of this
     tree and of TREE alternated, and bench.py --dump-outputs of both compared file by file.

Prints one JSON object (median / min / max of each number, the card and its power limit) and
writes it to --out when given.

    python tools/reset_envs_bench.py --rounds 5 --out profiles/r8_reset_envs_bench.json --parent ../parent
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from env_params_bench import card, engine  # noqa: E402  pylint: disable=wrong-import-position


def stats(values):
    r = np.array(values, dtype=np.float64)
    return {'median': float(np.median(r)), 'min': float(r.min()), 'max': float(r.max()), 'runs': [float(x) for x in r]}


def engine_stream(physics):
    import torch
    ptr = ctypes.c_void_p()
    physics._check(physics.lib.fb_device_ptr_stream(physics._handle, ctypes.byref(ptr)))  # pylint: disable=protected-access
    return torch.cuda.ExternalStream(ptr.value, device=0)


def restart_costs(args):
    """(1): device ms of one fb_reset_envs_where per mask size, host ms of one fb_reset."""
    import torch
    physics, model, (qpos0, qvel0) = engine('salamander_swim', args.swim_envs, args.ring)
    stream = engine_stream(physics)
    n = physics.n_envs
    q0 = torch.as_tensor(qpos0, dtype=torch.float32, device='cuda')
    v0 = torch.as_tensor(qvel0, dtype=torch.float32, device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(3)
    masks = {}
    for label, count in (('1', 1), ('1%', n//100), ('10%', n//10), ('100%', n)):
        mask = torch.zeros(n, dtype=torch.bool, device='cuda')
        mask[torch.randperm(n, device='cuda', generator=gen)[:count]] = True
        masks[label] = mask
    physics.reset(qpos0, qvel0)
    physics.step(args.inner)
    times = {label: [] for label in masks}
    times['fb_reset (host, whole batch)'] = []
    for _ in range(args.rounds):
        for label, mask in masks.items():
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            physics.synchronize()
            with torch.cuda.stream(stream):
                ev0.record()
                for _ in range(args.repeat):
                    physics.reset_envs(mask, q0, v0)
                ev1.record()
            physics.synchronize()
            times[label].append(ev0.elapsed_time(ev1)/args.repeat)
        physics.synchronize()
        t0 = time.perf_counter()
        physics.reset(qpos0, qvel0)
        times['fb_reset (host, whole batch)'].append(1e3*(time.perf_counter() - t0))
        assert not physics.flags.any()
    physics.close()
    return {'n_envs': n, 'unit': 'ms per call', 'repeat': args.repeat,
            'configs': {k: dict(stats(v), masked=int(masks[k].sum()) if k in masks else n) for k, v in times.items()}}


def clock_costs(args):
    """(2): env-steps/s with the episode clock unbound / bound, alternated."""
    import torch
    from env_params_bench import timed
    out = {}
    for key, name, n in (('swim', 'salamander_swim', args.swim_envs), ('ground', 'salamander', args.ground_envs)):
        physics, _, (qpos0, qvel0) = engine(name, n, args.ring)
        stream = engine_stream(physics)
        one = np.zeros(n, bool)
        one[n//2] = True
        rates = {'unbound': [], 'bound': []}
        for _ in range(args.rounds):
            for cfg in rates:
                physics.reset(qpos0, qvel0)
                if cfg == 'bound':
                    physics.step(args.inner)
                    physics.reset_envs(one, qpos0)
                rates[cfg].append(timed(physics, stream, args.inner, args.launches, args.warmup))
                assert not (physics.flags & 1).any(), f'{key}/{cfg}: non-finite state'
        base = float(np.median(rates['unbound']))
        for cfg, r in rates.items():
            out[f'{key}/{cfg}'] = dict(stats(r), n_envs=n, cost_vs_unbound_percent=float(100.0*(1.0 - np.median(r)/base)))
        physics.close()
        torch.cuda.synchronize()
    return {'unit': 'env-steps/s', 'launches_per_window': args.launches, 'physics_steps_per_launch': args.inner,
            'configs': out}


def headline(args):
    """(3): bench.py of this tree and of the parent alternated; --dump-outputs compared."""
    trees = {'this': ROOT, 'parent': os.path.abspath(args.parent)}
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--steps', str(args.bench_steps), '--warmup', '3']
    lines = {k: [] for k in trees}
    for _ in range(args.bench_rounds):
        for key, tree in trees.items():
            res = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, check=True)
            line = [ln for ln in res.stdout.splitlines() if ln.startswith('{')][-1]
            lines[key].append(json.loads(line))
    out = {'command': ' '.join(cmd[1:]), 'lines': lines}
    for metric in ('value', 'env_steps_per_s', 'throughput'):
        if all(metric in ln for v in lines.values() for ln in v):
            out['metric'] = metric
            out.update({k: stats([ln[metric] for ln in v]) for k, v in lines.items()})
            break
    with tempfile.TemporaryDirectory() as tmp:
        dirs = {}
        for key, tree in trees.items():
            dirs[key] = os.path.join(tmp, key)
            subprocess.run(cmd[:2] + ['--gpus', '1', '--steps', '20', '--warmup', '3', '--dump-outputs', dirs[key]],
                           cwd=tree, capture_output=True, text=True, check=True)
        files = sorted(os.listdir(dirs['this']))
        same = {}
        for f in files:
            a, b = np.load(os.path.join(dirs['this'], f)), np.load(os.path.join(dirs['parent'], f))
            same[f] = bool(a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes())
        out['dump_outputs_bit_identical'] = same
        out['dump_outputs_parent_files'] = sorted(os.listdir(dirs['parent']))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n', 1)[0])
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--repeat', type=int, default=20, help='restarts per timed window')
    ap.add_argument('--launches', type=int, default=30, help='timed launches per throughput window')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--inner', type=int, default=16, help='physics steps per launch')
    ap.add_argument('--ring', type=int, default=64)
    ap.add_argument('--swim-envs', type=int, default=65536)
    ap.add_argument('--ground-envs', type=int, default=4096)
    ap.add_argument('--parent', default=None, help='built checkout of the parent commit (for 3)')
    ap.add_argument('--bench-rounds', type=int, default=3)
    ap.add_argument('--bench-steps', type=int, default=100)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('reset_envs_bench.py: no CUDA device')
    out = {'card': card(), 'rounds': args.rounds, 'restart': restart_costs(args), 'episode_clock': clock_costs(args)}
    if args.parent:
        out['headline'] = headline(args)
    out['card_after'] = card()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
