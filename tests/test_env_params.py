"""Per-environment joint stiffness, joint damping, drag coefficients and water velocity
(fb_set_env_param, BatchedPhysics.set_env_params).

Environment e of a batch with per-environment tables must step as the fp64 oracle on the model
edited to e's values.  The emulation tests run the device code on the host (conftest.emu_library);
the ``-m gpu`` tests run the same checks, the kernel variants and the bit-for-bit comparison with a
homogeneous batch on a B200.
"""

import copy

import numpy as np
import pytest

from conftest import make_case, oracle_rollout, parity_errors

FIELDS = ('jnt_stiffness', 'dof_damping', 'drag_coefficients', 'water_velocity')


def env_values(model, tables, n_envs, seed=7, fields=FIELDS):
    """Distinct values of every field per environment: non-zero stiffness on every hinge (the
    models' own stiffness is zero, so the per-environment gate is what switches the spring on),
    scaled damping and drag coefficients, a water flow per environment.  The free joint keeps 0."""
    rng = np.random.default_rng(seed)
    hinge = np.asarray(model.jnt_type) != 0
    dof_free = np.asarray(model.jnt_type)[np.asarray(model.dof_jntid)] == 0
    out = {}
    if 'jnt_stiffness' in fields:
        out['jnt_stiffness'] = np.where(hinge, rng.uniform(0.005, 0.05, size=(n_envs, model.njnt)), 0.0)
    if 'dof_damping' in fields:
        base = np.asarray(model.dof_damping, dtype=np.float64)
        out['dof_damping'] = np.where(dof_free, 0.0, base*rng.uniform(0.2, 4.0, size=(n_envs, model.nv)))
    n_swim = len(tables.swim_links_index)
    if n_swim and 'drag_coefficients' in fields:
        base = np.asarray(tables.swim_coefficients, dtype=np.float64).reshape(n_swim, 2, 3)
        out['drag_coefficients'] = base*rng.uniform(0.3, 3.0, size=(n_envs, n_swim, 2, 3))
    if n_swim and 'water_velocity' in fields:
        out['water_velocity'] = rng.uniform(-0.2, 0.2, size=(n_envs, 3))
    return out


def edited(model, tables, values, env):
    """copy.deepcopy of model and tables with environment env's values written in."""
    model, tables = copy.deepcopy(model), copy.deepcopy(tables)
    if 'jnt_stiffness' in values:
        model.jnt_stiffness = np.array(values['jnt_stiffness'][env], dtype=np.float64)
    if 'dof_damping' in values:
        model.dof_damping = np.array(values['dof_damping'][env], dtype=np.float64)
    if 'drag_coefficients' in values:
        shape = np.shape(tables.swim_coefficients)
        tables.swim_coefficients = np.array(values['drag_coefficients'][env], dtype=np.float64).reshape(shape)
    if 'water_velocity' in values:
        tables.water_velocity = np.array(values['water_velocity'][env], dtype=np.float64)
    return model, tables


def oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps):
    """Worst parity error of each array over `envs`, each against the oracle on its edited model."""
    qpos, qvel, logs = physics.qpos, physics.qvel, physics.log_arrays()
    assert not (physics.flags[list(envs)] & 3).any(), physics.flags
    worst = {}
    for env in envs:
        m, t = edited(model, physics.tables, values, env)
        _, data, states = oracle_rollout(spec, m, t, n_steps + 1, qpos0[env], qvel0[env], ctrl[env])
        errs = parity_errors(qpos[env], qvel[env], {k: v[env] for k, v in logs.items()}, *states[-1], data)
        errs.pop('detail')
        for key, val in errs.items():
            worst[key] = max(worst.get(key, 0.0), val)
    return worst


def run_batch(library, name, n_envs, n_steps, fields=FIELDS, path='fast', seed=0, setup=None):
    """One batch with env_values tables of `fields`, stepped n_steps on one kernel path: 'fast'
    (per-thread kernels, the default), 'fast_team' (per-thread unconstrained kernel, team kernel on
    the hand-overs) or 'team' (team kernel only).  Returns the case, the tables and the batch."""
    from farms_mujoco_b200.engine import BatchedPhysics
    spec, model, qpos0, qvel0, ctrl = make_case(name, n_envs, seed=seed)
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=library)
    if path == 'team':
        physics.set_fast_path(False)
    elif path == 'fast_team':
        physics.set_constraint_path(False)
    if setup:
        setup(physics)
    values = env_values(model, physics.tables, n_envs, fields=fields)
    physics.set_env_params(**values)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    return (spec, model, qpos0, qvel0, ctrl), values, physics


# ----------------------------------------------------------------------------------- API
def test_api_validation_and_read_back(emu_library):
    from farms_mujoco_b200.engine import BatchedPhysics, EngineError
    spec, model, qpos0, qvel0, _ = make_case('salamander_swim', 3)
    physics = BatchedPhysics.from_spec(spec, 3, buffer_size=2, library=emu_library)
    n_swim = len(physics.tables.swim_links_index)
    # nothing set: the model's values, broadcast
    got = physics.env_params()
    assert got['jnt_stiffness'].shape == (3, model.njnt) and got['dof_damping'].shape == (3, model.nv)
    assert got['drag_coefficients'].shape == (3, n_swim, 2, 3) and got['water_velocity'].shape == (3, 3)
    assert np.array_equal(got['dof_damping'], np.tile(model.dof_damping, (3, 1)))
    assert np.array_equal(got['drag_coefficients'],
                          np.broadcast_to(np.reshape(physics.tables.swim_coefficients, (n_swim, 2, 3)), (3, n_swim, 2, 3)))
    assert np.array_equal(got['water_velocity'], np.tile(physics.tables.water_velocity, (3, 1)))

    def refused(match, **kw):
        with pytest.raises(EngineError, match=match):
            physics.set_env_params(**kw)

    stiff = np.zeros((3, model.njnt))
    stiff[:, 1:] = 0.01
    bad = stiff.copy()
    bad[2, 5] = -1.0
    refused(r'FB_ENV_JNT_STIFFNESS.*negative value at environment 2, index 5', jnt_stiffness=bad)
    bad = stiff.copy()
    bad[1, 3] = np.nan
    refused(r'FB_ENV_JNT_STIFFNESS.*non-finite value at environment 1, index 3', jnt_stiffness=bad)
    bad = stiff.copy()
    bad[0, 0] = 0.5
    refused(r'FB_ENV_JNT_STIFFNESS.*free joint.*environment 0, index 0', jnt_stiffness=bad)
    damp = np.tile(model.dof_damping, (3, 1))
    bad = damp.copy()
    bad[1, 4] = 0.1
    refused(r'FB_ENV_DOF_DAMPING.*free joint.*environment 1, index 4', dof_damping=bad)
    bad = damp.copy()
    bad[0, 10] = np.inf
    refused(r'FB_ENV_DOF_DAMPING.*environment 0, index 10', dof_damping=bad)
    bad = damp.copy()
    bad[2, 7] = -0.01
    refused(r'FB_ENV_DOF_DAMPING.*negative value at environment 2, index 7', dof_damping=bad)
    coef = -np.ones((3, n_swim, 2, 3))           # FARMS drag coefficients are negative
    coef[1, 3, 1, 2] = np.nan
    refused(r'FB_ENV_DRAG_COEF.*non-finite value at environment 1, index 23', drag_coefficients=coef)
    refused(r'FB_ENV_WATER_VELOCITY.*non-finite.*environment 0, index 1', water_velocity=[0.1, np.nan, 0.0])
    with pytest.raises(ValueError, match='jnt_stiffness'):
        physics.set_env_params(jnt_stiffness=np.zeros(model.njnt + 1))
    with pytest.raises(TypeError, match='unknown field'):
        physics.set_env_params(stiffness=stiff)
    # nothing of the refused calls was kept
    assert np.array_equal(physics.env_params()['jnt_stiffness'], np.zeros((3, model.njnt)))

    # broadcasting, read-back, only the keywords passed change, negative water velocity is a flow
    physics.set_env_params(jnt_stiffness=stiff[0], water_velocity=[-0.1, 0.05, 0.0])
    got = physics.env_params()
    assert np.array_equal(got['jnt_stiffness'], stiff)
    assert np.array_equal(got['water_velocity'], np.tile([-0.1, 0.05, 0.0], (3, 1)))
    with pytest.raises(EngineError, match='fb_set_water_velocity.*FB_ENV_WATER_VELOCITY'):
        physics.set_water_velocity([0.1, 0.0, 0.0])
    damp2 = damp*np.array([[1.0], [2.0], [3.0]])
    physics.set_env_params(dof_damping=damp2)
    got = physics.env_params()
    assert np.array_equal(got['dof_damping'], damp2) and np.array_equal(got['jnt_stiffness'], stiff)
    # tables survive reset
    physics.reset(qpos0, qvel0)
    got = physics.env_params()
    assert np.array_equal(got['dof_damping'], damp2) and np.array_equal(got['water_velocity'][1], [-0.1, 0.05, 0.0])
    # None restores the model value; fb_set_water_velocity is accepted again
    physics.set_env_params(water_velocity=None, jnt_stiffness=None)
    got = physics.env_params()
    assert np.array_equal(got['jnt_stiffness'], np.tile(model.jnt_stiffness, (3, 1)))
    assert np.array_equal(got['dof_damping'], damp2)
    physics.set_water_velocity([0.1, 0.0, 0.0])
    assert np.array_equal(physics.env_params()['water_velocity'], np.tile([0.1, 0.0, 0.0], (3, 1)))
    physics.close()


def test_drag_fields_need_swimming_links(emu_library):
    from farms_mujoco_b200.engine import BatchedPhysics, EngineError
    spec, model, *_ = make_case('salamander', 2)
    physics = BatchedPhysics.from_spec(spec, 2, buffer_size=2, library=emu_library)
    if len(physics.tables.swim_links_index):
        pytest.skip('model has swimming links')
    with pytest.raises(EngineError, match='FB_ENV_WATER_VELOCITY.*no swimming links'):
        physics.set_env_params(water_velocity=[0.1, 0.0, 0.0])
    with pytest.raises(EngineError, match='FB_ENV_DRAG_COEF.*no swimming links'):
        physics.set_env_params(drag_coefficients=np.ones((2, 0, 2, 3)))
    physics.close()


def test_cleared_tables_are_bit_identical(emu_library):
    """Tables set and then cleared leave the default path: the same bits as a batch that never set one."""
    from farms_mujoco_b200.engine import BatchedPhysics
    spec, model, qpos0, qvel0, ctrl = make_case('salamander_swim', 3)
    out = []
    for clear in (False, True):
        physics = BatchedPhysics.from_spec(spec, 3, buffer_size=5, library=emu_library)
        if clear:
            physics.set_env_params(**env_values(model, physics.tables, 3))
            physics.set_env_params(**dict.fromkeys(FIELDS))
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(4)
        out.append((physics.qpos, physics.log_arrays()))
    assert np.array_equal(out[0][0], out[1][0])
    for kind in out[0][1]:
        assert np.array_equal(out[0][1][kind], out[1][1][kind]), kind


# -------------------------------------------------------------------- oracle parity (host)
@pytest.mark.parametrize('name,path,n_steps,tol', [
    ('salamander_swim', 'fast', 12, 2e-5),     # per-thread unconstrained kernel
    ('salamander', 'fast', 8, 2e-5),           # ground: per-thread constrained kernel (fastc)
    ('salamander_swim', 'team', 12, 5e-4),     # team kernel
    ('salamander', 'team', 8, 5e-3),
])
def test_oracle_parity_emulated(emu_library, name, path, n_steps, tol):
    case, values, physics = run_batch(emu_library, name, 4, n_steps, path=path)
    spec, model, qpos0, qvel0, ctrl = case
    if name == 'salamander':
        assert set(values) == {'jnt_stiffness', 'dof_damping'}
        if path == 'fast':
            assert physics.last_pending == 4            # the constrained kernel stepped them
    else:
        assert set(values) == set(FIELDS)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, range(4), n_steps)
    print(name, path, {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < (5e-4 if key == 'contacts' and path == 'fast' else tol), (key, val, worst)


def test_env_stiffness_pulls_to_cpg_spring_references(emu_library):
    """On-device CPG driving spring references: with a per-environment stiffness the joints are
    pulled to the reference of each step of the sequence -- the batch equals, environment by
    environment, batches of the model edited to that environment's stiffness."""
    import dataclasses
    import re
    import fastpath_cases
    from farms_mujoco_b200 import models
    from farms_mujoco_b200.simulation.simulation import Simulation
    spring_joints = ('joint_5', 'joint_6')
    n_envs, n_it, chunk = 2, 24, 8
    stiffness = (0.03, 0.12)

    def run(mjcf_stiffness, table):
        spec = models.swimmer8(n_iterations=n_it)
        mjcf, count = re.subn(r'(<joint name="joint_[56]"[^>]*?)stiffness="0.0"',
                              rf'\1stiffness="{mjcf_stiffness}"', spec.mjcf)
        assert count == 2
        spec = dataclasses.replace(spec, mjcf=mjcf)
        sim = Simulation.from_spec(spec, n_envs=n_envs, chunk=chunk, library=emu_library,
                                   controller=fastpath_cases.swimmer_cpg(n_envs, True, spring_joints=spring_joints))
        if table is not None:
            sim.physics.set_env_params(jnt_stiffness=table)
        sim.run()
        return sim.task.data.sensors.joints.array.copy(), sim.physics.qpos_spring

    # the model's stiffness is zero on every joint: the tables alone switch the springs on
    from farms_mujoco_b200.mjcf_subset import parse_mjcf
    model = parse_mjcf(models.swimmer8().mjcf)
    jids = [list(model.jnt_names).index(j) for j in spring_joints]
    table = np.zeros((n_envs, model.njnt))
    for e in range(n_envs):
        table[e, jids] = stiffness[e]
    mixed, springs = run('0.0', table)
    free, _ = run('0.0', None)
    assert np.abs(springs[:, 7 + 5:]).max() > 0.05                   # the references moved
    for e in range(n_envs):
        ref, _ = run(str(stiffness[e]), None)
        err = np.abs(mixed[e] - ref[e]).max()/max(1e-2, np.abs(ref[e]).max())   # [n_envs, it, joint, col]
        assert err < 2e-5, (e, err)
        # ... and the spring acts: without it the joints move otherwise
        assert np.abs(free[e, :, :, 0] - ref[e, :, :, 0]).max() > 1e-4


# ----------------------------------------------------------------------------------- B200
# The same oracle parity on every kernel path and variant, the mixed batch against homogeneous
# batches of the edited models, and the headline batch size with every field set.
SAMPLE = (0, 1, 31, 32, 33)


@pytest.mark.gpu
@pytest.mark.parametrize('lean', [True, False])
@pytest.mark.parametrize('name,path,n_envs,n_steps', [
    ('salamander_swim', 'fast', 64, 12),        # small batch: SPLIT variant of the unconstrained kernel
    ('salamander_swim', 'fast_team', 64, 12),
    ('salamander_swim', 'team', 64, 12),
    ('salamander', 'fast', 64, 8),              # ground: constrained kernel and its SPLIT variant
    ('salamander', 'fast_team', 64, 8),
    ('salamander', 'team', 64, 8),
])
def test_gpu_oracle_parity(cuda_library, name, path, n_envs, n_steps, lean):
    case, values, physics = run_batch(cuda_library, name, n_envs, n_steps, path=path,
                                      setup=lambda p: p.set_fast_lean(lean))
    spec, model, qpos0, qvel0, ctrl = case
    if path != 'team':
        assert physics.fast_path and physics.last_pending == (0 if name == 'salamander_swim' else n_envs)
    print(name, path, 'lean' if lean else 'general', 'split', physics.fast_split, 'con_split', physics.con_split)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, SAMPLE + (n_envs - 1,), n_steps)
    print({k: f'{v:.2e}' for k, v in worst.items()})
    team = path == 'team' or (path == 'fast_team' and name == 'salamander')
    for key, val in worst.items():
        tol = (5e-3 if key == 'contacts' else 5e-4) if team else (5e-4 if key == 'contacts' else 2e-5)
        assert val < tol, (key, val, worst)


@pytest.mark.gpu
@pytest.mark.parametrize('slim', [1, 7])
def test_gpu_oracle_parity_slim(cuda_library, slim, monkeypatch):
    """SLIM layout, one warp per block and MULTI (7 warps kept in step), at 8,192 environments."""
    monkeypatch.setenv('FARMS_B200_FAST_BLOCK', '32')            # SLIM needs full warps
    n_envs, n_steps = 8192, 8
    case, values, physics = run_batch(cuda_library, 'salamander_swim', n_envs, n_steps,
                                      setup=lambda p: p.set_fast_slim(slim))
    assert physics.fast_slim == slim and physics.last_pending == 0
    spec, model, qpos0, qvel0, ctrl = case
    envs = (0, 31, 32, 32*slim - 1, 32*slim, n_envs//2 + 5, n_envs - 1)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps)
    print('slim', slim, {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < 2e-5, (key, val, worst)


@pytest.mark.gpu
def test_gpu_hand_over_mid_launch(cuda_library):
    """Swimming environments meet a joint limit after a few steps (a different step in every
    environment, some never): the unconstrained ENVP = 1 kernel hands them over to the constrained one."""
    import fastpath_cases
    from farms_mujoco_b200.engine import BatchedPhysics
    n_envs, n_steps = 70, 16
    spec, model, qpos0, qvel0, ctrl = fastpath_cases.hand_over_case('salamander_swim', n_envs)
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=cuda_library)
    values = env_values(model, physics.tables, n_envs, fields=('dof_damping', 'drag_coefficients', 'water_velocity'))
    physics.set_env_params(**values)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    pending = physics.last_pending
    assert 0 < pending < n_envs, pending
    envs = (0, 1, n_envs//2, n_envs - 2, n_envs - 1)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps)
    print('hand-over', pending, {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < 5e-5, (key, val, worst)


def homogeneous_physics(library, spec, model, values, env, n_envs, n_steps):
    """A batch of the model edited to environment env's values, every field in the model itself
    (no table): the default entry points."""
    from farms_mujoco_b200.engine import BatchedPhysics
    spec = copy.deepcopy(spec)
    m, _ = edited(model, None, {k: v for k, v in values.items() if k in ('jnt_stiffness', 'dof_damping')}, env)
    swim = [link for link in spec.animat_options.morphology.links if link.swimming]
    if 'drag_coefficients' in values:
        for i, link in enumerate(swim):
            link.drag_coefficients = np.array(values['drag_coefficients'][env][i]).tolist()
    if 'water_velocity' in values:
        spec.arena_options.water.velocity = np.array(values['water_velocity'][env]).tolist()
    physics = BatchedPhysics(m, n_envs, spec.links_names, spec.joints_names, spec.contacts_names, spec.xfrc_names,
                             animat_options=spec.animat_options, arena_options=spec.arena_options,
                             units=spec.simulation_options.units, buffer_size=n_steps + 1, library=library)
    got = physics.env_params()
    for key, val in values.items():
        assert np.array_equal(got[key][0], val[env]), key
    return physics


@pytest.mark.gpu
@pytest.mark.parametrize('name,path,n_envs,slim', [
    ('salamander_swim', 'fast', 64, 0),       # SPLIT variant
    ('salamander_swim', 'fast', 8192, 7),     # SLIM + MULTI
    ('salamander', 'fast', 64, 0),            # constrained kernel
    ('salamander_swim', 'team', 64, 0),
])
def test_gpu_mixed_batch_equals_homogeneous_batches(cuda_library, name, path, n_envs, slim, monkeypatch):
    """Environment e of a batch with per-environment tables (the ENVP = 1 kernels) against a batch of
    the model edited to e's values (the default entry points), same kernel variant, same inputs in
    every environment: the same bits, or a few ulp where ptxas contracts the ENVP = 1 kernels differently."""
    from farms_mujoco_b200.engine import BatchedPhysics
    if slim:
        monkeypatch.setenv('FARMS_B200_FAST_BLOCK', '32')        # SLIM needs full warps
    n_steps = 8
    spec, model, qpos0, qvel0, ctrl = make_case(name, 1)
    qpos0, qvel0, ctrl = (np.repeat(a, n_envs, axis=0) for a in (qpos0, qvel0, ctrl))

    def run(physics):
        physics.set_fast_path(path != 'team')
        if slim:
            physics.set_fast_slim(slim)
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(n_steps)
        logs = physics.log_arrays()
        return physics.qpos, physics.qvel, logs

    mixed = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=cuda_library)
    values = env_values(model, mixed.tables, n_envs)
    mixed.set_env_params(**values)
    mq, mv, mlogs = run(mixed)
    identical, worst = True, 0.0
    for env in (0, 5, n_envs - 1):
        hq, hv, hlogs = run(homogeneous_physics(cuda_library, spec, model, values, env, n_envs, n_steps))
        pairs = [(mq[env], hq[env]), (mv[env], hv[env])] + [(mlogs[k][env], hlogs[k][env]) for k in mlogs]
        for a, b in pairs:
            identical &= np.array_equal(a, b)
            if a.size:
                worst = max(worst, float(np.abs(a.astype(np.float64) - b).max()/max(1e-30, np.abs(b).max())))
    print(name, path, n_envs, 'bit-identical' if identical else f'differs by {worst:.1e} (relative)')
    assert worst < 1e-5, worst


@pytest.mark.gpu
def test_gpu_full_batch_all_fields(cuda_library):
    """65,536 SALAMANDERs in water, 16 steps in one launch (bench.py's headline configuration:
    synthetic inputs, on-device travelling wave) with all four fields set: no flags, and sampled
    environments within the bench configuration's tolerance of the oracle on their edited models."""
    from farms_mujoco_b200 import models, mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.models import travelling_wave_parameters
    from farms_mujoco_b200.sharding import synthetic_inputs
    from oracle.oracle import OraclePhysics
    from oracle import farms_oracle as fo
    from conftest import log_errors, state_errors
    n_envs, n_steps = 65536, 16
    spec = models.MODELS['salamander_swim']()
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    qpos0, qvel0, phase = synthetic_inputs(model, np.arange(n_envs))
    joints, amp, freq, lag = travelling_wave_parameters(spec)
    acts = [model.actuator_id(f'actuator_position_{j}') for j in joints]
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=cuda_library)
    physics.set_env_phase(phase)
    physics.set_wave_controller(acts, amp, freq, lag)
    values = env_values(model, physics.tables, n_envs)
    physics.set_env_params(**values)
    physics.reset(qpos0, qvel0)
    assert physics.fast_slim == 7
    physics.step(n_steps)
    assert not physics.flags.any() and physics.last_pending == 0
    rng = np.random.default_rng(3)
    sample = sorted({0, 31, 32, 223, 224, n_envs//2, n_envs - 1} | set(int(e) for e in rng.integers(0, n_envs, size=5)))
    qpos, qvel = physics.qpos, physics.qvel
    worst = {}
    for env in sample:
        def controller(iteration, time, env=env):
            ctrl = np.zeros(model.nu)
            ctrl[acts] = amp*np.sin(2*np.pi*freq*time - lag + phase[env])
            return ctrl
        m, t = edited(model, physics.tables, values, env)
        data, states = fo.reference_rollout(OraclePhysics(m), spec, t, n_steps + 1, controller=controller,
                                            qpos0=qpos0[env], qvel0=qvel0[env])
        ours = physics.export_farms(env)
        for key, val in state_errors(qpos[env], qvel[env], *states[-1]).items():
            worst[key] = max(worst.get(key, 0.0), val)
        for kind in ('links', 'joints', 'contacts', 'xfrc'):
            ref = getattr(data.sensors, kind).array
            for key, val in log_errors(kind, getattr(ours.sensors, kind).array, ref).items():
                worst[f'{kind}.{key}'] = max(worst.get(f'{kind}.{key}', 0.0), val)
    print('65536 envs, all fields:', {k: f'{v:.1e}' for k, v in worst.items() if v > 0})
    for key, val in worst.items():
        assert val < 5e-5, (key, val, worst)
