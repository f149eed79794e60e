"""Frictionless <contact><pair> self-collisions (the reference writes every self-collision with
friction=[0]*5, mjcf.py:1012-1033; MuJoCo floors that at mu = 1e-5) under
parse_mjcf(..., frictionless_pairs='hard'): one hard normal row per contact with the normal force as
a multiplier, solved in the team kernel (fb_device.h, DESIGN.md section 8).

The fp64 oracle keeps solving the reference's model, the soft pyramidal rows of kind 20
(mjcf_subset.soft_pair_model).  The hard row drops terms of relative size mu: the states, the normal
forces and the contact sensors' reaction and total columns are held to the tolerances of the other
pair tests (2e-4); the sensors' friction columns differ from the oracle's by the tangential force of a
mu = 1e-5 cone, at most mu times the normal force, and are held to that bound instead."""

import dataclasses

import numpy as np
import pytest

from conftest import PARITY_FLOOR, oracle_rollout, parity_errors

PAIR = ('link_leg_0_L_3', 'link_leg_0_R_3')
TOL = 2e-4
# Groups of the two 100-step held-pose cases held to a looser bound, with the errors measured on the
# emulation build (group-wise relative, conftest.PARITY_FLOOR) and their cause:
#  'swim': a resting leg joint keeps a period-2 oscillation (the sign of its velocity flips every
#    step, ~0.01 rad/s) in the oracle and here alike.  The mu = 1e-5 tangential force the hard row
#    drops -- 1.7e-5 N on a 2 g foot, an impulse of ~8.5e-6 m/s a step against a foot speed of ~1e-4
#    m/s -- damps it: it decays by 0.6 % a step in the oracle, 0.3 % here.  After 100 steps: joint
#    velocity 2.5e-1 (2.5e-3 rad/s absolute on velocities below 1e-2 rad/s, while the joint angles
#    agree to 3.6e-6 rad), joints.velocity 1.4e-3, links.velocity_ang 9.6e-4, links.velocity_lin 4.6e-4.
#  'ground': the limit force of the trunk joint held at its limit, 1.1e-3.  (The mu = 0.5 pairs of the
#    dense-Hessian path reach 4.5e-4 on the joint velocities of the same pose.)
LOOSE = {
    'swim': {'joint_velocity': 0.5, 'joints.velocity': 5e-3, 'links.velocity_ang': 4e-3, 'links.velocity_lin': 4e-3,
             'root_velocity_ang': 1e-3},
    'ground': {'joints.limit_force': 4e-3, 'joint_velocity': 1e-3, 'joints.velocity': 1e-3, 'links.velocity_ang': 1e-3,
               'links.velocity_lin': 1e-3},
}


def _hard_spec(swimming=True, mixed=False):
    import variant_models
    spec = variant_models.salamander_foot_pairs(swimming=swimming, friction=0)
    if mixed:
        # the hind girdle's pair with mu = 0.5: a soft pair (kind 20) beside a hard one (kind 21)
        old = 'geom2="link_leg_1_R_3_foot" condim="3" friction="0 0 0 0 0"'
        assert spec.mjcf.count(old) == 1
        spec = dataclasses.replace(spec, mjcf=spec.mjcf.replace(
            old, 'geom2="link_leg_1_R_3_foot" condim="3" friction="0.5 0.5 0 0 0"'))
    return spec


def _pair_inputs(model, n, seed=5, apart_last=True):
    """_pair_case of test_emu_parity.py: legs folded (feet of each girdle pressed together), random
    joint offsets, velocities and controls; the last environment with the legs apart."""
    import variant_models
    rng = np.random.default_rng(seed)
    qpos0 = np.tile(variant_models.folded_legs_qpos(model, 1.0), (n, 1))
    qpos0[:, 7:] += rng.uniform(-0.03, 0.03, (n, model.nq - 7))
    if apart_last:
        qpos0[n - 1] = model.key_qpos
    qvel0 = rng.uniform(-0.2, 0.2, (n, model.nv))
    ctrl = rng.uniform(-0.3, 0.3, (n, model.nu))
    return qpos0, qvel0, ctrl


def _held_inputs(model, n, seed=0, spread=0.005):
    """Legs held folded (joint angles within `spread` of the fold): the position actuators' targets
    are the initial joint angles (tools/pair_bench.py), the bodies start at rest."""
    import variant_models
    rng = np.random.default_rng(seed)
    qpos0 = np.tile(variant_models.folded_legs_qpos(model, 1.0), (n, 1))
    qpos0[:, 7:] += rng.uniform(-spread, spread, (n, model.nq - 7))
    qvel0 = np.zeros((n, model.nv))
    ctrl = np.zeros((n, model.nu))
    for j in range(model.njnt):
        act = f'actuator_position_{model.jnt_names[j]}'
        if act in model.actuator_names:
            ctrl[:, model.actuator_names.index(act)] = qpos0[:, model.jnt_qposadr[j]]
    return qpos0, qvel0, ctrl


def _run(library, spec, qpos0, qvel0, ctrl, n_steps):
    from farms_mujoco_b200.engine import BatchedPhysics
    physics = BatchedPhysics.from_spec(spec, len(qpos0), buffer_size=n_steps + 1, library=library,
                                       frictionless_pairs='hard')
    assert physics.fast_path == 0                          # two-body rows: team kernel only
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    return physics


def compare_hard_with_oracle(spec, model, physics, qpos0, qvel0, ctrl, envs, n_steps, tol=TOL, loose=None):
    """compare_with_oracle (fastpath_cases.py) against the oracle on the reference's soft model, every
    group at `tol` (or its bound in `loose`) except the contact sensors' friction columns: those are
    bounded by the tangential force the hard row drops, mu (1e-5) times the largest normal force of
    the pairs, plus `tol`."""
    loose = loose or {}
    from farms_mujoco_b200 import mjcf_subset
    assert not physics.flags.any(), physics.flags          # no non-finite state, no unsettled solve
    reference = mjcf_subset.soft_pair_model(model)
    qpos, qvel, logs = physics.qpos, physics.qvel, physics.log_arrays()
    names = [tuple(c) for c in spec.contacts_names]
    pairs = [k for k, c in enumerate(names) if c[1]]
    worst = {}
    for env in envs:
        _, data, states = oracle_rollout(spec, reference, physics.tables, n_steps + 1, qpos0[env], qvel0[env], ctrl[env])
        errs = parity_errors(qpos[env], qvel[env], {k: v[env] for k, v in logs.items()}, *states[-1], data)
        detail = errs['detail']
        ref = data.sensors.contacts.array
        ours = logs['contacts'][env]
        dropped = mjcf_subset.MJ_MINMU*np.abs(ref[:, pairs, 0:3]).max()
        fric = np.abs(ours[..., 3:6] - ref[..., 3:6]).max()
        scale = max(np.abs(ref[..., 3:6]).max(), PARITY_FLOOR)
        detail['contacts.friction'] = max(0.0, fric - dropped)/scale
        for key, val in detail.items():
            worst[key] = max(worst.get(key, 0.0), val)
    print(spec.name, n_steps, 'steps:', {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < loose.get(key, tol), (key, val, worst)
    return worst


# ---- front-end ---------------------------------------------------------------------------------

def test_hard_option_compiles_frictionless_pairs(monkeypatch):
    """'hard': the two frictionless foot pairs become kind 21 with mu at MuJoCo's floor; geometry,
    solref, solimp, margin and gap are what kind 20 gets (compiled with the floor check lifted)."""
    from farms_mujoco_b200 import mjcf_subset
    spec = _hard_spec()
    hard = mjcf_subset.parse_mjcf(spec.mjcf, frictionless_pairs='hard')
    sel = hard.cand_end == 21
    assert sel.sum() == 2 and (hard.cand_end == 20).sum() == 0
    assert np.all(hard.cand_friction[sel] == mjcf_subset.MJ_MINMU)
    monkeypatch.setattr(mjcf_subset, 'PAIR_MIN_FRICTION', 0.0)
    soft = mjcf_subset.parse_mjcf(spec.mjcf)
    assert np.array_equal(np.where(sel, 20, hard.cand_end), soft.cand_end)
    for name in ('cand_geom1', 'cand_geom2', 'cand_friction', 'cand_solref', 'cand_solimp', 'cand_margin', 'cand_gap'):
        assert np.array_equal(getattr(hard, name), getattr(soft, name)), name
    assert np.array_equal(mjcf_subset.soft_pair_model(hard).cand_end, soft.cand_end)


def test_hard_option_still_refuses_low_friction():
    """mu = 0.05 is not frictionless: dropping a 5 % tangential force is not the stated approximation."""
    import variant_models
    from farms_mujoco_b200 import mjcf_subset
    with pytest.raises(NotImplementedError, match='friction') as err:
        mjcf_subset.parse_mjcf(variant_models.salamander_foot_pairs(friction=0.05).mjcf, frictionless_pairs='hard')
    assert 'frictionless_pairs' not in str(err.value)


def test_frictionless_pairs_option_values():
    from farms_mujoco_b200 import mjcf_subset
    with pytest.raises(ValueError, match='frictionless_pairs'):
        mjcf_subset.parse_mjcf(_hard_spec().mjcf, frictionless_pairs='soft')
    # the default refuses and names the option
    with pytest.raises(NotImplementedError, match="friction.*frictionless_pairs='hard'"):
        mjcf_subset.parse_mjcf(_hard_spec().mjcf)


# ---- the oracle: the yardstick did not move ------------------------------------------------------

def test_oracle_pin_soft_pair_model(emu_library, monkeypatch):
    """The oracle on soft_pair_model(hard model) is the oracle on the kind-20 model the reference
    compiles: bit-identical rollouts, pair contacts included."""
    from farms_mujoco_b200 import mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    spec = _hard_spec()
    hard = mjcf_subset.parse_mjcf(spec.mjcf, frictionless_pairs='hard')
    tables = BatchedPhysics.from_spec(spec, 1, library=emu_library, frictionless_pairs='hard').tables
    monkeypatch.setattr(mjcf_subset, 'PAIR_MIN_FRICTION', 0.0)
    soft = mjcf_subset.parse_mjcf(spec.mjcf)
    qpos0, qvel0, ctrl = _pair_inputs(hard, 2)
    outs = []
    for model in (soft, mjcf_subset.soft_pair_model(hard)):
        _, data, states = oracle_rollout(spec, model, tables, 9, qpos0[0], qvel0[0], ctrl[0])
        outs.append((states, {k: getattr(data.sensors, k).array.copy() for k in ('links', 'joints', 'contacts')}))
    (sa, la), (sb, lb) = outs
    assert len(sa) == len(sb) and all(np.array_equal(x, y) for st_a, st_b in zip(sa, sb) for x, y in zip(st_a, st_b))
    assert all(np.array_equal(la[k], lb[k]) for k in la)
    names = [tuple(c) for c in spec.contacts_names]
    assert np.abs(la['contacts'][1:, names.index(PAIR), 0:3]).max() > 1e-3       # the pair is in contact


# ---- cases: emulation build here, the device below ------------------------------------------------

def _case(kind, n):
    """(spec, model, qpos0, qvel0, ctrl, n_steps) of one parity case.
    'pair': the _pair_case of test_emu_parity.py, 12 steps, the last environment with the legs apart;
    'swim': legs held folded in water, 100 steps; 'ground': the same on the ground (plane contacts)
    with a trunk joint held at its limit, where the feet part and meet again; 'mixed': the 'pair' inputs on a model whose hind pair has
    mu = 0.5 (kind 20, dense Hessian) beside the frictionless front pair (kind 21)."""
    from farms_mujoco_b200 import mjcf_subset
    spec = _hard_spec(swimming=kind != 'ground', mixed=kind == 'mixed')
    model = mjcf_subset.parse_mjcf(spec.mjcf, frictionless_pairs='hard')
    if kind in ('pair', 'mixed'):
        return (spec, model) + _pair_inputs(model, n) + (12,)
    qpos0, qvel0, ctrl = _held_inputs(model, n)
    if kind == 'ground':
        qpos0[:, 7 + 3] = 1.004                           # a trunk joint past its limit, held there
        for j in range(model.njnt):
            act = f'actuator_position_{model.jnt_names[j]}'
            if act in model.actuator_names:
                ctrl[:, model.actuator_names.index(act)] = qpos0[:, model.jnt_qposadr[j]]
    return spec, model, qpos0, qvel0, ctrl, 100


def check_case(library, kind, n, envs):
    spec, model, qpos0, qvel0, ctrl, n_steps = _case(kind, n)
    if kind == 'mixed':
        assert (model.cand_end == 20).sum() == 1 and (model.cand_end == 21).sum() == 1
    physics = _run(library, spec, qpos0, qvel0, ctrl, n_steps)
    logs = physics.log_arrays()
    contacts = logs['contacts']
    names = [tuple(c) for c in spec.contacts_names]
    pairs = [names.index((f'link_leg_{i}_L_3', f'link_leg_{i}_R_3')) for i in range(2)]
    if kind in ('pair', 'mixed'):
        # the feet push on one another (which environments and girdles depends on the seeded
        # velocities, drawn for the whole batch: the oracle agrees, compared below)
        force = np.abs(contacts[:, 1:, pairs, 6:9]).max(axis=(1, 3))          # [env, pair]
        assert (force[:n - 1] > 1e-3).any(axis=0).all(), force                 # each pair in some environment
        assert (force[:n - 1].max(axis=1) > 1e-3).mean() > 0.5, force          # a pair in most of them
        assert not contacts[n - 1, :, pairs].any()                            # legs apart: nothing
    else:
        active = np.abs(contacts[:, 1:, pairs, 0:3]).max(axis=-1) > 0
        if kind == 'swim':
            # both pair contacts active in every step in most environments.  A resting frictionless
            # contact settles at dist = margin, on the detection threshold, and rounding drops it for a
            # step now and then -- in the fp64 reference as well, at steps its own rounding decides
            assert active.all(axis=(1, 2)).mean() > 0.7, active.all(axis=(1, 2))
        else:
            # on the ground the feet part and meet again (at the same steps as in the oracle: the
            # comparison below) -- the pair contacts are made and broken under load
            assert active.mean() > 0.5 and not active.all(), active.mean()
        if kind == 'ground':
            from farms_mujoco_b200.layout import sc
            plane = [k for k, c in enumerate(names) if not c[1]]
            assert (np.abs(contacts[:, 1:, plane, 0:3]).max(axis=(-2, -1)) > 0).all()
            assert (np.abs(logs['joints'][:, 1:, :, sc.joint_limit_force]).max(axis=(1, 2)) > 0).all()   # a limit row
    # sensors: (g1, g2) and (g1, -1) on the left link, (g2, -1) with the opposite sign on the right
    # (sensors.pyx:160-176); the hard row carries no tangential force
    left, right = names.index((PAIR[0], '')), names.index((PAIR[1], ''))
    if kind != 'ground':             # on the ground the feet's sensors also see the plane
        assert np.allclose(contacts[:, :, pairs[0], 6:9], contacts[:, :, left, 6:9], atol=1e-6)
        assert np.allclose(contacts[:, :, pairs[0], 6:9], -contacts[:, :, right, 6:9], atol=1e-6)
    normal = np.abs(contacts[:, :, pairs[0], 0:3]).max()
    assert np.abs(contacts[:, :, pairs[0], 3:6]).max() <= 1e-6*normal
    return compare_hard_with_oracle(spec, model, physics, qpos0, qvel0, ctrl, envs, n_steps, loose=LOOSE.get(kind))


@pytest.mark.parametrize('kind,n', [('pair', 3), ('swim', 2), ('ground', 2), ('mixed', 3)])
def test_frictionless_pairs_vs_oracle(emu_library, kind, n):
    check_case(emu_library, kind, n, range(n))


def test_self_collisions_from_sdf_hard(emu_library):
    """morphology.self_collisions through Simulation.from_sdf with frictionless_pairs='hard': the
    reference's frictionless pair runs.  The legs of the branching walker stand close enough for the
    feet to overlap and swing sideways (hips about x), so the pair pushes them apart against the
    position actuators."""
    from farms_mujoco_b200.options import (AnimatOptions, ArenaOptions, ControlOptions, MorphologyOptions,
                                           MotorOptions, SimulationOptions, SpawnOptions)
    from farms_mujoco_b200.simulation.simulation import Simulation
    from test_sdf_subset import branching_sdf
    sdf = branching_sdf()
    for old, new in (('<link name="leg_L"><pose>0.05 0.04 0 ', '<link name="leg_L"><pose>0.05 0.009 0 '),
                     ('<link name="leg_R"><pose>0.05 -0.04 0 ', '<link name="leg_R"><pose>0.05 -0.009 0 '),
                     ('<xyz>0.0 1.0 0.0</xyz>', '<xyz>1.0 0.0 0.0</xyz>'),
                     ('<child>leg_R</child>\n    <axis><xyz>0 1 0</xyz>', '<child>leg_R</child>\n    <axis><xyz>1 0 0</xyz>')):
        assert sdf.count(old) == 1, old
        sdf = sdf.replace(old, new)
    animat = AnimatOptions(sdf=sdf, spawn=SpawnOptions(pose=[0, 0, 0.06, 0, 0, 0]),
                           morphology=MorphologyOptions(self_collisions=[['leg_L', 'leg_R']]),
                           control=ControlOptions(motors=[MotorOptions(joint_name=j, gains=[0.5, 1e-3])
                                                          for j in ('spine', 'hip_L', 'hip_R')]))
    contacts_names = [('trunk_0', ''), ('trunk_1', ''), ('leg_L', ''), ('leg_R', ''), ('leg_L', 'leg_R')]
    sim = Simulation.from_sdf(SimulationOptions(timestep=1e-3, n_iterations=60), animat, ArenaOptions(ground_height=0.0),
                              n_envs=2, library=emu_library, frictionless_pairs='hard', contacts_names=contacts_names)
    assert sim.physics.fast_path == 0
    sim.run()
    sensors = sim.task.data.sensors
    assert np.isfinite(sensors.links.array).all() and np.isfinite(sim.physics.qpos).all()
    assert not sim.physics.flags.any()
    pair = sensors.contacts.array[..., 4, :]
    assert np.abs(pair[..., 0:3]).max() > 1e-4                           # the feet push on one another
    assert np.abs(pair[..., 3:6]).max() <= 1e-6*np.abs(pair[..., 0:3]).max()


# ---- the device --------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['pair', 'swim', 'ground', 'mixed'])
def test_frictionless_pairs_on_device(cuda_library, kind):
    """The four cases above on the B200 (team kernel, TEAM = 32) with 40 environments; no environment
    flagged (non-finite state, contact overflow, unsettled hard-row solve)."""
    from farms_mujoco_b200.engine import BatchedPhysics
    n = 40
    spec, model, qpos0, qvel0, ctrl, n_steps = _case(kind, n)
    physics = BatchedPhysics.from_spec(spec, n, buffer_size=2, library=cuda_library, frictionless_pairs='hard')
    assert physics.team_lanes > 1
    del physics
    check_case(cuda_library, kind, n, (0, 1, 17, n - 2, n - 1))
