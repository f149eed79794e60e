"""Cost of the per-environment actuator gain and bias tables (set_env_params(actuator_gainprm=...,
actuator_biasprm=...)) on the step kernels.

Alternates, round after round in one process, device-timed windows of
  swim/none    65,536 SALAMANDERs in water, 16 steps a launch, travelling wave on (bench.py's
               headline configuration: LEAN kernel, FT_HAS_WAVE)
  swim/act     the same with a gain and a bias table (kp / kv x0.5 .. x2 per environment)
  ground/none  4,096 SALAMANDERs on the ground (every step constrained)
  ground/act   the same with both tables
so that every configuration sees the same machine state; the tables of one engine are set and
cleared between its windows.  Prints one JSON object (median / min / max env-steps/s of each
configuration, the cost against its table-free run, the card, its power limit and the SM clock read
after the timed rounds) and writes it to --out when given.

    python tools/env_actuators_bench.py --rounds 5 --launches 30 --out profiles/r9_env_actuators_bench.json
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from env_params_bench import card, engine, timed  # noqa: E402  pylint: disable=wrong-import-position


def sm_clock():
    """Current SM clock and power draw of GPU 0 (read-only query)."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=clocks.sm,power.draw', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        clock, power = [s.strip() for s in out.split(',')]
        return {'sm_clock': clock, 'power_draw': power}
    except Exception as exc:  # pylint: disable=broad-except
        return {'sm_clock': f'unknown ({exc})'}


def act_tables(model, n_envs, seed=11):
    """A kp / kv sweep around the model's values: position and velocity actuators x0.5 .. x2."""
    rng = np.random.default_rng(seed)
    gain0 = np.asarray(model.actuator_gainprm, dtype=np.float64)[:, 0]
    bias0 = np.asarray(model.actuator_biasprm, dtype=np.float64)[:, :3]
    scale = rng.uniform(0.5, 2.0, size=(n_envs, model.nu))
    scale[:, (bias0[:, 1] == 0) & (bias0[:, 2] == 0)] = 1.0          # motors keep theirs
    return {'actuator_gainprm': gain0*scale, 'actuator_biasprm': bias0*scale[..., None]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n', 1)[0])
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--launches', type=int, default=30, help='timed launches per window')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--inner', type=int, default=16, help='physics steps per launch')
    ap.add_argument('--ring', type=int, default=64)
    ap.add_argument('--swim-envs', type=int, default=65536)
    ap.add_argument('--ground-envs', type=int, default=4096)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('env_actuators_bench.py: no CUDA device')
    specs = {'swim': ('salamander_swim', args.swim_envs), 'ground': ('salamander', args.ground_envs)}
    configs = [('swim', 'none'), ('swim', 'act'), ('ground', 'none'), ('ground', 'act')]
    out = {'card': card(), 'rounds': args.rounds, 'launches_per_window': args.launches,
           'physics_steps_per_launch': args.inner, 'ring': args.ring, 'unit': 'env-steps/s', 'configs': {}}
    engines = {key: engine(name, n, args.ring) for key, (name, n) in specs.items()}
    streams, tables = {}, {}
    for key, (physics, model, _) in engines.items():
        ptr = ctypes.c_void_p()
        physics._check(physics.lib.fb_device_ptr_stream(physics._handle, ctypes.byref(ptr)))  # pylint: disable=protected-access
        streams[key] = torch.cuda.ExternalStream(ptr.value, device=0)
        tables[key] = act_tables(model, physics.n_envs)
    rates = {f'{e}/{c}': [] for e, c in configs}
    for _ in range(args.rounds):
        for eng, cfg in configs:
            physics, _, (qpos0, qvel0) = engines[eng]
            physics.set_env_params(**{f: (v if cfg == 'act' else None) for f, v in tables[eng].items()})
            physics.reset(qpos0, qvel0)
            rates[f'{eng}/{cfg}'].append(timed(physics, streams[eng], args.inner, args.launches, args.warmup))
            assert not physics.flags.any(), f'{eng}/{cfg}: flags set'
    out['card'].update(sm_clock())
    for eng, cfg in configs:
        r = np.array(rates[f'{eng}/{cfg}'])
        base = np.median(rates[f'{eng}/none'])
        physics, model = engines[eng][:2]
        width = 4*model.nu + 6*model.njnt if cfg == 'act' else 0       # gain, bias and the derived linear forms
        out['configs'][f'{eng}/{cfg}'] = {
            'n_envs': physics.n_envs, 'median': float(np.median(r)), 'min': float(r.min()), 'max': float(r.max()),
            'spread_percent': float(100.0*(r.max() - r.min())/np.median(r)), 'runs': [float(x) for x in r],
            'cost_vs_none_percent': float(100.0*(1.0 - np.median(r)/base)),
            'table_bytes': int(4*width*physics.log_view.env_pad),
        }
    for physics, _, _ in engines.values():
        physics.close()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
