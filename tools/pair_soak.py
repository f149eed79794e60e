"""Soak of the pair-contact path (team kernel, dense Newton Hessian): SALAMANDERs with explicit
foot-foot <pair>s, the legs driven around the folded pose so that the feet meet and part again,
on the ground (plane contacts and pair contacts in one solve).  With --frictionless: the reference's
frictionless pairs, solved as hard normal rows (frictionless_pairs='hard').
usage: python tools/pair_soak.py <n_envs> <launches of 16 steps> [library] [--frictionless]"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import variant_models  # noqa: E402
from farms_mujoco_b200 import mjcf_subset  # noqa: E402
from farms_mujoco_b200.engine import BatchedPhysics  # noqa: E402

frictionless = '--frictionless' in sys.argv
args = [a for a in sys.argv[1:] if a != '--frictionless']
n, launches = int(args[0]), int(args[1])
library = args[2] if len(args) > 2 else None
fp = 'hard' if frictionless else 'refuse'
# (in water the folded pose itself goes unstable after ~400 steps -- in the fp64 oracle too: explicit
# Euler under the legs' drag -- so the soak runs on the ground, plane and pair contacts in one solve)
for swimming in (False,):
    spec = variant_models.salamander_foot_pairs(swimming=swimming, **({'friction': 0} if frictionless else {}))
    model = mjcf_subset.parse_mjcf(spec.mjcf, frictionless_pairs=fp)
    rng = np.random.default_rng(0)
    fold = variant_models.folded_legs_qpos(model, 1.0)
    qpos0 = np.tile(fold, (n, 1))
    qpos0[:, 7:] += rng.uniform(-0.03, 0.03, (n, model.nq - 7))
    ph = BatchedPhysics.from_spec(spec, n, buffer_size=17, library=library, frictionless_pairs=fp)
    ph.reset(qpos0, None)
    names = [tuple(c) for c in spec.contacts_names]
    pair = [i for i, c in enumerate(names) if c[1]]
    ctrl = np.zeros((n, model.nu))
    acts = {}
    for j in range(model.njnt):
        act = f'actuator_position_{model.jnt_names[j]}'
        if act in model.actuator_names:
            acts[model.actuator_names.index(act)] = model.jnt_qposadr[j]
    phase = rng.uniform(0, 2*np.pi, n)
    t0 = time.time()
    made = broken = 0
    was = np.zeros(n, dtype=bool)
    for k in range(launches):
        # legs open and close by 4 .. 12 % around the folded pose, 2 Hz, per-environment amplitude
        swing = (0.04 + 0.08*phase/(2*np.pi))*np.sin(2*np.pi*2.0*k*16*model.timestep)
        for a, adr in acts.items():
            ctrl[:, a] = fold[adr]*(1.0 - swing) if abs(fold[adr]) > 0.5 else fold[adr]
        ph.set_ctrl(ctrl)
        ph.step(16)
        now = np.abs(ph.log_row('contacts', 16 if k == 0 else (16*(k + 1)) % 17)[:, pair, 6:9]).max(axis=(1, 2)) > 0
        made += int((now & ~was).sum())
        broken += int((~now & was).sum())
        was = now
    f = ph.flags
    print('salamander_foot_pairs' + (' frictionless (hard rows)' if frictionless else ''), 'water' if swimming else 'ground', n, 'envs', launches*16, 'steps', 'sec %.2f' % (time.time() - t0),
          'nonfinite', int(np.count_nonzero(f & 1)), 'solver', int(np.count_nonzero(f & 4)),
          'pair contacts made', made, 'broken', broken, 'finite state', bool(np.isfinite(ph.qpos).all()),
          'max|qvel| %.2f' % np.abs(ph.qvel).max())
