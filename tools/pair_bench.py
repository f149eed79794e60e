"""Throughput of the team kernel on a model with explicit <pair> self-collisions (dense Newton
Hessian while a pair contact is active), on the same model with the reference's frictionless pairs
solved as hard normal rows (frictionless_pairs='hard', tree-sparse Hessian), and on the same pose
without the pairs, device-timed in one process.
usage: python tools/pair_bench.py [n_envs]"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import variant_models  # noqa: E402
from farms_mujoco_b200 import mjcf_subset, models  # noqa: E402
from farms_mujoco_b200.engine import BatchedPhysics  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
inner, launches = 16, 6
out = {'n_envs': n, 'steps_per_launch': inner, 'launches': launches}
try:
    out['gpu'] = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                                capture_output=True, text=True, check=True).stdout.strip()
except (OSError, subprocess.CalledProcessError):
    out['gpu'] = 'unknown'
for name, spec, fast, fp in (
        ('salamander_foot_pairs (team kernel, pair contacts active)', variant_models.salamander_foot_pairs(), None, 'refuse'),
        ('salamander_foot_pairs frictionless, hard normal rows (team kernel, pair contacts active)',
         variant_models.salamander_foot_pairs(friction=0), None, 'hard'),
        ('salamander_swim forced onto the team kernel, same pose', models.salamander(swimming=True), 0, 'refuse')):
    model = mjcf_subset.parse_mjcf(spec.mjcf, frictionless_pairs=fp)
    rng = np.random.default_rng(0)
    qpos0 = np.tile(variant_models.folded_legs_qpos(model, 1.0), (n, 1))
    qpos0[:, 7:] += rng.uniform(-0.03, 0.03, (n, model.nq - 7))
    ph = BatchedPhysics.from_spec(spec, n, buffer_size=inner + 1, frictionless_pairs=fp)
    if fast is not None:
        ph.set_fast_path(fast)
    # hold the folded pose: the position actuators' targets are the initial joint angles
    ctrl = np.zeros((n, model.nu))
    for j in range(model.njnt):
        act = f'actuator_position_{model.jnt_names[j]}'
        if act in model.actuator_names:
            ctrl[:, model.actuator_names.index(act)] = qpos0[:, model.jnt_qposadr[j]]
    ph.reset(qpos0, None)
    ph.set_ctrl(ctrl)
    ph.step(inner)
    ms = []
    for _ in range(launches):
        ph.step(inner)
        ms.append(ph.last_step_ms())
    pair = [i for i, c in enumerate(spec.contacts_names) if c[1]]
    active = float((np.abs(ph.log_row('contacts', inner)[:, pair, 6:9]).max(axis=(1, 2)) > 0).mean()) if pair else 0.0
    out[name] = {'ms_per_launch': float(np.median(ms)), 'env_steps_per_s': n*inner/(np.median(ms)*1e-3),
                 'team_lanes': ph.team_lanes, 'fast_path': ph.fast_path, 'envs_flagged': int(np.count_nonzero(ph.flags)),
                 'envs_with_an_active_pair_contact_in_the_last_row': active}
print(json.dumps(out, indent=1))
