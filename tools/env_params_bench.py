"""Cost of the per-environment parameter tables (BatchedPhysics.set_env_params) on the step kernels.

Alternates, round after round in one process, device-timed windows of
  swim/none    65,536 SALAMANDERs in water, 16 steps a launch (bench.py's headline configuration)
  swim/drag    the same with per-environment drag coefficients
  swim/all     the same with all four fields (stiffness, damping, drag coefficients, water velocity)
  swim/friction  the headline batch with per-environment contact friction (the swimming path does
               not read it: the unconstrained kernels keep their entry points)
  ground/none  4,096 SALAMANDERs on the ground (every step constrained)
  ground/sd    the same with per-environment stiffness and damping
  ground/friction  the same with per-environment contact friction
  ground/all   friction, stiffness and damping
  centipede/none, centipede/friction  8,192 CENTIPEDEs on the ground, without and with friction
so that every configuration sees the same machine state (the CENTIPEDE pair alternates in a group of
its own, after the SALAMANDER engines are closed); the tables of one engine are set and cleared
between its windows.  Prints one JSON object (median / min / max env-steps/s of each
configuration, the cost against its table-free run, the card and its power limit) and writes it to
--out when given.

    python tools/env_params_bench.py --rounds 5 --launches 30 --out profiles/r7_env_friction_bench.json
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    """Name, power limit and maximum SM clock of GPU 0 (read-only query)."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader',
                              '-i', '0'], capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(',')]
        return {'name': name, 'power_limit': power, 'sm_max_clock': clock}
    except Exception as exc:  # pylint: disable=broad-except
        import torch
        return {'name': torch.cuda.get_device_name(0), 'power_limit': f'unknown ({exc})'}


def table_values(model, tables, n_envs, fields, seed=11):
    """Distinct per-environment values of `fields`, near the model's own (a sweep around it)."""
    rng = np.random.default_rng(seed)
    hinge = np.asarray(model.jnt_type) != 0
    dof_free = np.asarray(model.jnt_type)[np.asarray(model.dof_jntid)] == 0
    n_swim = len(tables.swim_links_index)
    out = {}
    if 'jnt_stiffness' in fields:
        out['jnt_stiffness'] = np.where(hinge, rng.uniform(0.0, 0.02, size=(n_envs, model.njnt)), 0.0)
    if 'dof_damping' in fields:
        out['dof_damping'] = np.where(dof_free, 0.0, np.asarray(model.dof_damping)*rng.uniform(0.5, 2.0, size=(n_envs, model.nv)))
    if 'drag_coefficients' in fields:
        base = np.asarray(tables.swim_coefficients, dtype=np.float64).reshape(n_swim, 2, 3)
        out['drag_coefficients'] = base*rng.uniform(0.5, 2.0, size=(n_envs, n_swim, 2, 3))
    if 'water_velocity' in fields:
        out['water_velocity'] = rng.uniform(-0.05, 0.05, size=(n_envs, 3))
    if 'geom_friction' in fields:
        out['geom_friction'] = rng.uniform(0.5, 1.5, size=(n_envs, model.ngeom))
    return out


def table_width(model, field, values):
    """Device table entries per environment: one per collision candidate for the friction."""
    return model.ncand if field == 'geom_friction' else int(np.prod(values.shape[1:]))


def engine(name, n_envs, ring):
    from farms_mujoco_b200 import models, mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.models import travelling_wave_parameters
    from farms_mujoco_b200.sharding import synthetic_inputs
    spec = models.MODELS[name]()
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    qpos0, qvel0, phase = synthetic_inputs(model, np.arange(n_envs))
    joints, amp, freq, lag = travelling_wave_parameters(spec)
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=ring)
    physics.set_env_phase(phase)
    physics.set_wave_controller([model.actuator_id(f'actuator_position_{j}') for j in joints], amp, freq, lag)
    return physics, model, (qpos0, qvel0)


def timed(physics, stream, inner, launches, warmup):
    import torch
    for _ in range(warmup):
        physics.step(inner, sync=False)
    physics.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record()
        for _ in range(launches):
            physics.step(inner, sync=False)
        ev1.record()
    physics.synchronize()
    return physics.n_envs*inner*launches/(ev0.elapsed_time(ev1)*1e-3)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n', 1)[0])
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--launches', type=int, default=30, help='timed launches per window')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--inner', type=int, default=16, help='physics steps per launch')
    ap.add_argument('--ring', type=int, default=64)
    ap.add_argument('--swim-envs', type=int, default=65536)
    ap.add_argument('--ground-envs', type=int, default=4096)
    ap.add_argument('--centipede-envs', type=int, default=8192)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('env_params_bench.py: no CUDA device')
    all_fields = ('jnt_stiffness', 'dof_damping', 'drag_coefficients', 'water_velocity', 'geom_friction')
    # Two groups, each alternated round after round: the SALAMANDER engines, then the CENTIPEDE
    # engine once they are closed.  A kernel's shared-memory limit is an attribute of the function,
    # which every engine of the process shares, and a SALAMANDER engine's block-size review sets it
    # for its smaller model: the CENTIPEDE's launches need the engines of the other model gone.
    groups = [
        ({'swim': ('salamander_swim', args.swim_envs), 'ground': ('salamander', args.ground_envs)},
         [('swim', 'none', ()), ('swim', 'drag', ('drag_coefficients',)),
          ('swim', 'all', all_fields[:4]), ('swim', 'friction', ('geom_friction',)),
          ('ground', 'none', ()), ('ground', 'sd', ('jnt_stiffness', 'dof_damping')),
          ('ground', 'friction', ('geom_friction',)),
          ('ground', 'all', ('geom_friction', 'jnt_stiffness', 'dof_damping'))]),
        ({'centipede': ('centipede', args.centipede_envs)},
         [('centipede', 'none', ()), ('centipede', 'friction', ('geom_friction',))]),
    ]
    out = {'card': card(), 'rounds': args.rounds, 'launches_per_window': args.launches,
           'physics_steps_per_launch': args.inner, 'ring': args.ring, 'unit': 'env-steps/s', 'configs': {}}
    for specs, configs in groups:
        engines = {key: engine(name, n, args.ring) for key, (name, n) in specs.items()}
        streams, tables = {}, {}
        for key, (physics, model, _) in engines.items():
            ptr = ctypes.c_void_p()
            physics._check(physics.lib.fb_device_ptr_stream(physics._handle, ctypes.byref(ptr)))  # pylint: disable=protected-access
            streams[key] = torch.cuda.ExternalStream(ptr.value, device=0)
            tables[key] = table_values(model, physics.tables, physics.n_envs, all_fields)
        rates = {f'{e}/{c}': [] for e, c, _ in configs}
        for _ in range(args.rounds):
            for eng, cfg, fields in configs:
                physics, _, (qpos0, qvel0) = engines[eng]
                physics.set_env_params(**{f: (tables[eng][f] if f in fields else None) for f in all_fields})
                physics.reset(qpos0, qvel0)
                rates[f'{eng}/{cfg}'].append(timed(physics, streams[eng], args.inner, args.launches, args.warmup))
                assert not physics.flags.any(), f'{eng}/{cfg}: flags set'
        for eng, cfg, fields in configs:
            r = np.array(rates[f'{eng}/{cfg}'])
            base = np.median(rates[f'{eng}/none'])
            physics = engines[eng][0]
            width = sum(table_width(physics.model, f, tables[eng][f]) for f in fields)
            table_bytes = 4*width*physics.log_view.env_pad
            out['configs'][f'{eng}/{cfg}'] = {
                'n_envs': physics.n_envs, 'fields': list(fields), 'median': float(np.median(r)), 'min': float(r.min()),
                'max': float(r.max()), 'runs': [float(x) for x in r],
                'cost_vs_none_percent': float(100.0*(1.0 - np.median(r)/base)),
                'table_bytes': int(table_bytes),
                'table_bytes_per_env_step': 4*width,
                'log_bytes_per_env_step': physics.log_bytes_per_env_step,
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
