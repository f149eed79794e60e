"""Per-environment actuator gains and biases (fb_set_env_param FB_ENV_ACT_GAIN / FB_ENV_ACT_BIAS,
BatchedPhysics.set_env_params(actuator_gainprm=..., actuator_biasprm=...)).

Environment e of a batch with gain / bias tables must step as the fp64 oracle on the model with e's
``actuator_gainprm[:, 0]`` and ``actuator_biasprm[:, 0:3]`` written in.  The emulation tests run the
device code on the host (conftest.emu_library); the ``-m gpu`` tests run the same checks on every
kernel variant the launch plan can pick, and the bit-for-bit comparison with homogeneous batches.
"""

import copy

import numpy as np
import pytest

from conftest import make_case, parity_errors
from test_env_params import SAMPLE, edited, env_values

ACT_FIELDS = ('actuator_gainprm', 'actuator_biasprm')


def act_values(model, n_envs, seed=11):
    """Random motor gains per environment and actuator: kp x0.3 .. x3 on the position actuators
    (gain kp, bias [0, -kp, 0]), kv x0.3 .. x2 on the velocity actuators (gain kv, bias [0, 0, -kv];
    the models' kv sit well inside the explicit Euler bound kv*dt/I < 2, models.py), and on the
    motors a gain x0.5 .. x2 and a small constant bias torque."""
    rng = np.random.default_rng(seed)
    gain0 = np.asarray(model.actuator_gainprm, dtype=np.float64)[:, 0]
    bias0 = np.asarray(model.actuator_biasprm, dtype=np.float64)[:, :3]
    pos, vel = bias0[:, 1] != 0, bias0[:, 2] != 0
    scale = np.where(vel, rng.uniform(0.3, 2.0, (n_envs, model.nu)),
                     np.where(pos, rng.uniform(0.3, 3.0, (n_envs, model.nu)), rng.uniform(0.5, 2.0, (n_envs, model.nu))))
    bias = bias0*scale[..., None]
    bias[..., 0] = np.where(pos | vel, bias0[:, 0], rng.uniform(-0.01, 0.01, (n_envs, model.nu)))
    return {'actuator_gainprm': gain0*scale, 'actuator_biasprm': bias}


def edited_act(model, tables, values, env):
    """The model (and tables) with environment env's values of every field in `values` written in."""
    model, tables = edited(model, tables, values, env)
    model = copy.deepcopy(model)
    if 'actuator_gainprm' in values:
        g = np.array(model.actuator_gainprm, dtype=np.float64)
        g[:, 0] = values['actuator_gainprm'][env]
        model.actuator_gainprm = g
    if 'actuator_biasprm' in values:
        b = np.array(model.actuator_biasprm, dtype=np.float64)
        b[:, :3] = values['actuator_biasprm'][env]
        model.actuator_biasprm = b
    return model, tables


def wave_of(spec, model):
    """The travelling wave of bench.py's headline: actuators, amplitude, frequency, phase lag."""
    from farms_mujoco_b200.models import travelling_wave_parameters
    joints, amp, freq, lag = travelling_wave_parameters(spec)
    return [model.actuator_id(f'actuator_position_{j}') for j in joints], amp, freq, lag


def oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps, wave=None):
    """Worst parity error of each array over `envs`, each against the oracle on its edited model
    (physics.model: it carries the forcerange edits of set_actuator_forcerange)."""
    from oracle.oracle import OraclePhysics
    from oracle import farms_oracle as fo
    qpos, qvel, logs = physics.qpos, physics.qvel, physics.log_arrays()
    assert not (physics.flags[list(envs)] & 3).any(), physics.flags
    worst = {}
    for env in envs:
        def controller(iteration, time, env=env):
            c = np.array(ctrl[env], dtype=np.float64)
            if wave is not None:
                acts, amp, freq, lag = wave
                c[acts] = amp*np.sin(2*np.pi*freq*time - lag)
            return c
        m, t = edited_act(physics.model, physics.tables, values, env)
        data, states = fo.reference_rollout(OraclePhysics(m), spec, t, n_steps + 1, controller=controller,
                                            qpos0=qpos0[env], qvel0=qvel0[env])
        errs = parity_errors(qpos[env], qvel[env], {k: v[env] for k, v in logs.items()}, *states[-1], data)
        errs.pop('detail')
        for key, val in errs.items():
            worst[key] = max(worst.get(key, 0.0), val)
    return worst


def run_act_batch(library, spec, n_envs, n_steps, path='fast', wave=False, fields=(), setup=None, seed=0,
                  case=None):
    """One batch with act_values tables (plus env_values tables of `fields`), stepped n_steps on
    one kernel path: 'fast' (per-thread kernels), 'fast_team' (team kernel on the hand-overs) or
    'team'.  The tables are set before the wave controller, so the records are rebuilt under them."""
    from farms_mujoco_b200 import mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    if case is None:
        rng = np.random.default_rng(seed)
        qpos0 = np.tile(model.key_qpos, (n_envs, 1))
        qpos0[:, 7:] += rng.uniform(-0.1, 0.1, size=(n_envs, model.nq - 7))
        qvel0 = np.tile(model.key_qvel, (n_envs, 1)) + rng.uniform(-0.3, 0.3, size=(n_envs, model.nv))
        ctrl = rng.uniform(-0.3, 0.3, size=(n_envs, model.nu))
    else:
        qpos0, qvel0, ctrl = case
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=library)
    if path == 'team':
        physics.set_fast_path(False)
    elif path == 'fast_team':
        physics.set_constraint_path(False)
    if setup:
        setup(physics)
    values = act_values(model, n_envs)
    if fields:
        values.update(env_values(model, physics.tables, n_envs, fields=fields))
    physics.set_env_params(**values)
    w = None
    if wave:
        w = wave_of(spec, model)
        physics.set_wave_controller(*w)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    return (model, qpos0, qvel0, ctrl, w), values, physics


def spec_of(name):
    import variant_models
    from farms_mujoco_b200 import models
    return variant_models.swimmer8_features() if name == 'swimmer8_features' else models.MODELS[name]()


# ----------------------------------------------------------------------------------- API
def test_api_validation_and_read_back(emu_library):
    from farms_mujoco_b200.engine import BatchedPhysics, EngineError
    spec, model, qpos0, qvel0, _ = make_case('swimmer8', 3)
    physics = BatchedPhysics.from_spec(spec, 3, buffer_size=4, library=emu_library)
    nu = model.nu
    gain0 = np.asarray(model.actuator_gainprm, dtype=np.float64)[:, 0]
    bias0 = np.asarray(model.actuator_biasprm, dtype=np.float64)[:, :3]
    got = physics.env_params()
    assert got['actuator_gainprm'].shape == (3, nu) and got['actuator_biasprm'].shape == (3, nu, 3)
    assert np.array_equal(got['actuator_gainprm'], np.tile(gain0, (3, 1)))
    assert np.array_equal(got['actuator_biasprm'], np.broadcast_to(bias0, (3, nu, 3)))

    def refused(match, **kw):
        with pytest.raises(EngineError, match=match):
            physics.set_env_params(**kw)

    bad = np.tile(gain0, (3, 1))
    bad[1, 4] = np.nan
    refused(r'FB_ENV_ACT_GAIN.*non-finite value at environment 1, actuator 4', actuator_gainprm=bad)
    bad = np.tile(bias0, (3, 1, 1))
    bad[2, 6, 1] = -np.inf
    refused(r'FB_ENV_ACT_BIAS.*non-finite value at environment 2, actuator 6, column 1', actuator_biasprm=bad)
    with pytest.raises(ValueError, match='actuator_biasprm'):
        physics.set_env_params(actuator_biasprm=np.zeros((nu, 2)))
    assert np.array_equal(physics.env_params()['actuator_gainprm'], np.tile(gain0, (3, 1)))

    # no sign check (MuJoCo has none): a negative gain and a positive position bias are accepted
    gain = np.tile(gain0, (3, 1))*np.array([[1.0], [2.0], [-0.5]])
    physics.set_env_params(actuator_gainprm=gain, actuator_biasprm=-bias0)      # broadcast
    got = physics.env_params()
    assert np.array_equal(got['actuator_gainprm'], gain)
    assert np.array_equal(got['actuator_biasprm'], np.broadcast_to(-bias0, (3, nu, 3)))
    # tables survive reset and reset_envs
    physics.reset(qpos0, qvel0)
    physics.step(2)
    physics.reset_envs([1])
    got = physics.env_params()
    assert np.array_equal(got['actuator_gainprm'], gain)
    assert np.array_equal(got['actuator_biasprm'], np.broadcast_to(-bias0, (3, nu, 3)))
    # None restores the model's value of that field only
    physics.set_env_params(actuator_gainprm=None)
    got = physics.env_params()
    assert np.array_equal(got['actuator_gainprm'], np.tile(gain0, (3, 1)))
    assert np.array_equal(got['actuator_biasprm'], np.broadcast_to(-bias0, (3, nu, 3)))
    physics.set_env_params(actuator_biasprm=None)
    assert np.array_equal(physics.env_params()['actuator_biasprm'], np.broadcast_to(bias0, (3, nu, 3)))
    physics.close()


def test_cleared_tables_are_bit_identical(emu_library):
    """Gain and bias tables set and then cleared: the same bits as a batch that never set one."""
    from farms_mujoco_b200.engine import BatchedPhysics
    spec, model, qpos0, qvel0, ctrl = make_case('salamander_swim', 3)
    out = []
    for clear in (False, True):
        physics = BatchedPhysics.from_spec(spec, 3, buffer_size=5, library=emu_library)
        if clear:
            physics.set_env_params(**act_values(model, 3))
            physics.set_env_params(**dict.fromkeys(ACT_FIELDS))
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(4)
        out.append((physics.qpos, physics.qvel, physics.log_arrays()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    for kind in out[0][2]:
        assert np.array_equal(out[0][2][kind], out[1][2][kind]), kind


def test_derived_actuator_force(emu_library):
    """The reset's forward pass and the derived view (team kernel): actuator_force of each
    environment is its own gain * ctrl + bias0 + bias1 * q + bias2 * qd."""
    from farms_mujoco_b200.engine import BatchedPhysics
    n_envs = 4
    spec, model, qpos0, qvel0, ctrl = make_case('salamander', n_envs)
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=4, library=emu_library)
    values = act_values(model, n_envs)
    physics.set_env_params(**values)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(1, want_derived=True)
    got = physics.derived()['actuator_force']
    j = np.asarray(model.actuator_trnid)
    q = qpos0[:, np.asarray(model.jnt_qposadr)[j]]
    qd = qvel0[:, np.asarray(model.jnt_dofadr)[j]]
    b = values['actuator_biasprm']
    want = values['actuator_gainprm']*ctrl + b[..., 0] + b[..., 1]*q + b[..., 2]*qd
    err = np.abs(got - want).max()/np.abs(want).max()
    assert err < 1e-5, err
    # ... and they are not the model's
    base = np.asarray(model.actuator_gainprm)[:, 0]*ctrl + np.asarray(model.actuator_biasprm)[:, 1]*q + \
        np.asarray(model.actuator_biasprm)[:, 2]*qd
    assert np.abs(got - base).max() > 1e-2*np.abs(base).max()


# -------------------------------------------------------------------- oracle parity (host)
@pytest.mark.parametrize('name,path,wave,lean,n_steps,tol', [
    ('swimmer8', 'fast', True, True, 12, 2e-5),            # LEAN + FT_HAS_WAVE, chain
    ('salamander_swim', 'fast', True, True, 12, 2e-5),     # LEAN + FT_HAS_WAVE, SPLIT
    ('salamander_swim', 'fast', False, False, 12, 2e-5),   # general variant, linear form + load_joints
    ('salamander', 'fast', False, True, 8, 2e-5),          # ground: constrained kernel, hand-overs
    ('salamander', 'team', False, True, 8, 5e-3),          # team kernel
    ('swimmer8_features', 'fast', False, True, 12, 2e-5),  # clamped / geared actuators: actuation_generic
])
def test_oracle_parity_emulated(emu_library, name, path, wave, lean, n_steps, tol):
    n_envs = 4
    spec = spec_of(name)
    case, values, physics = run_act_batch(emu_library, spec, n_envs, n_steps, path=path, wave=wave,
                                          setup=lambda p: p.set_fast_lean(lean))
    model, qpos0, qvel0, ctrl, w = case
    if name == 'salamander' and path == 'fast':
        assert physics.last_pending == n_envs            # the constrained kernel stepped them
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, range(n_envs), n_steps, wave=w)
    print(name, path, 'wave' if wave else '', 'lean' if lean else 'general', {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < (5e-4 if key == 'contacts' and path == 'fast' else tol), (key, val, worst)


def test_with_other_fields_emulated(emu_library):
    """Gain and bias tables together with stiffness, damping and drag tables."""
    spec = spec_of('salamander_swim')
    case, values, physics = run_act_batch(emu_library, spec, 3, 10, wave=True,
                                          fields=('jnt_stiffness', 'dof_damping', 'drag_coefficients'))
    model, qpos0, qvel0, ctrl, w = case
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, range(3), 10, wave=w)
    for key, val in worst.items():
        assert val < 2e-5, (key, val, worst)


def test_forcerange_switch_rebuilds_derived_table(emu_library):
    """fb_set_actuator_forcerange after the tables are set: actuators switched off (initialize_control's
    [0, 0] range) contribute exactly zero and leave the derived linear forms; switched back on, they
    are in them again.  Each state against the oracle on the edited model."""
    from farms_mujoco_b200.engine import BatchedPhysics
    n_envs, n_steps = 3, 10
    spec, model, qpos0, qvel0, ctrl = make_case('salamander_swim', n_envs)
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=emu_library)
    values = act_values(model, n_envs)
    physics.set_env_params(**values)
    acts = [model.actuator_id(f'actuator_{k}_{j}') for j in spec.joints_names[:4] for k in ('position', 'velocity')]
    for off in (True, False):
        physics.set_actuator_forcerange(acts, [1 if off else 0]*len(acts), [[0.0, 0.0]]*len(acts))
        assert physics.fast_lean
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(n_steps)
        worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, range(n_envs), n_steps)
        print('off' if off else 'on', {k: f'{v:.2e}' for k, v in worst.items()})
        for key, val in worst.items():
            assert val < 2e-5, (key, val, worst)
        physics.step(1, want_derived=True)
        force = physics.derived()['actuator_force'][:, acts]
        if off:
            assert not force.any()
        else:
            assert (np.abs(force) > 0).all()


def test_cpg_sequence_with_env_gains(emu_library):
    """On-device CPG driving the position actuators (the per-step constants of a control sequence,
    seq_constants) with a kp per environment: environment by environment, the batch equals batches
    of the model with that environment's kp."""
    import dataclasses
    import re
    import fastpath_cases
    from farms_mujoco_b200 import models
    from farms_mujoco_b200.mjcf_subset import parse_mjcf
    from farms_mujoco_b200.simulation.simulation import Simulation
    n_envs, n_it, chunk = 2, 24, 8
    kps = (0.4, 2.5)

    def run(kp, table):
        spec = models.swimmer8(n_iterations=n_it)
        if kp is not None:
            mjcf, count = re.subn(r'(<position name="actuator_position_joint_\d+" joint="joint_\d+" kp=")1.0"',
                                  rf'\g<1>{kp!r}"', spec.mjcf)
            assert count == 7, count
            spec = dataclasses.replace(spec, mjcf=mjcf)
        sim = Simulation.from_spec(spec, n_envs=n_envs, chunk=chunk, library=emu_library,
                                   controller=fastpath_cases.swimmer_cpg(n_envs, True))
        if table is not None:
            sim.physics.set_env_params(**table)
        sim.run()
        return sim.task.data.sensors.joints.array.copy()

    model = parse_mjcf(models.swimmer8().mjcf)
    pos = [model.actuator_id(f'actuator_position_joint_{j}') for j in range(7)]
    gain = np.tile(np.asarray(model.actuator_gainprm, dtype=np.float64)[:, 0], (n_envs, 1))
    bias = np.tile(np.asarray(model.actuator_biasprm, dtype=np.float64)[:, :3], (n_envs, 1, 1))
    for e, kp in enumerate(kps):
        gain[e, pos] = kp
        bias[e, pos, 1] = -kp
    mixed = run(None, {'actuator_gainprm': gain, 'actuator_biasprm': bias})
    base = run(None, None)
    for e, kp in enumerate(kps):
        ref = run(kp, None)
        err = np.abs(mixed[e] - ref[e]).max()/max(1e-2, np.abs(ref[e]).max())
        assert err < 2e-5, (e, err)
        assert np.abs(base[e, :, :, 0] - ref[e, :, :, 0]).max() > 1e-4         # the gain acts


# ----------------------------------------------------------------------------------- B200
@pytest.mark.gpu
@pytest.mark.parametrize('lean', [True, False])
@pytest.mark.parametrize('name,path,wave,n_envs,n_steps,variant', [
    ('salamander_swim', 'fast', True, 64, 12, 'split'),        # SPLIT variant of the unconstrained kernel
    ('salamander_swim', 'fast', True, 64, 12, 'regular'),      # single-warp regular layout
    ('swimmer8', 'fast', True, 64, 12, 'regular'),
    ('salamander_swim', 'team', True, 64, 12, ''),
    ('salamander', 'fast', False, 64, 8, 'con_split'),         # ground: constrained SPLIT variant
    ('salamander', 'fast', False, 64, 8, 'con_single'),        # ... and the single-warp constrained kernel
    ('salamander', 'fast_team', False, 64, 8, ''),
    ('salamander', 'team', False, 64, 8, ''),
    ('swimmer8_features', 'fast', False, 64, 12, 'regular'),   # actuation_generic
])
def test_gpu_oracle_parity(cuda_library, name, path, wave, n_envs, n_steps, variant, lean):
    def setup(p):
        p.set_fast_lean(lean)
        if variant == 'regular':
            p.set_fast_split(False)
        if variant == 'con_single':
            p.set_con_split(False)
    spec = spec_of(name)
    case, values, physics = run_act_batch(cuda_library, spec, n_envs, n_steps, path=path, wave=wave, setup=setup)
    model, qpos0, qvel0, ctrl, w = case
    if path != 'team':
        assert physics.fast_path and physics.last_pending == (n_envs if name == 'salamander' else 0)
    if variant == 'split':
        assert physics.fast_split
    if variant == 'con_split':
        assert physics.con_split
    print(name, path, variant, 'lean' if lean else 'general', 'split', physics.fast_split, 'con_split', physics.con_split)
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, SAMPLE + (n_envs - 1,), n_steps, wave=w)
    print({k: f'{v:.2e}' for k, v in worst.items()})
    # the team kernel's ground-contact solver: 5e-3, its tolerance in test_emu_parity (the stiffer
    # gains of the sweep reach 1.4e-3 on qvel; test_gpu_mixed_batch_equals_homogeneous_batches shows
    # the team kernel bit-identical to a batch of the edited model, so this is the solver, not the tables)
    team = path == 'team' or (path == 'fast_team' and name == 'salamander')
    ground_team = team and name == 'salamander'
    for key, val in worst.items():
        tol = (5e-3 if key == 'contacts' or ground_team else 5e-4) if team else (5e-4 if key == 'contacts' else 2e-5)
        assert val < tol, (key, val, worst)


@pytest.mark.gpu
@pytest.mark.parametrize('slim', [1, 7])
def test_gpu_oracle_parity_slim(cuda_library, slim, monkeypatch):
    """SLIM layout, one warp per block and MULTI (7 warps kept in step), at 8,192 environments,
    with the travelling wave."""
    monkeypatch.setenv('FARMS_B200_FAST_BLOCK', '32')            # SLIM needs full warps
    n_envs, n_steps = 8192, 8
    spec = spec_of('salamander_swim')
    case, values, physics = run_act_batch(cuda_library, spec, n_envs, n_steps, wave=True,
                                          setup=lambda p: p.set_fast_slim(slim))
    assert physics.fast_slim == slim and physics.last_pending == 0
    model, qpos0, qvel0, ctrl, w = case
    envs = (0, 31, 32, 32*slim - 1, 32*slim, n_envs//2 + 5, n_envs - 1)
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps, wave=w)
    print('slim', slim, {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < 2e-5, (key, val, worst)


@pytest.mark.gpu
def test_gpu_hand_over_mid_launch(cuda_library):
    """Swimming environments meet a joint limit after a few steps (a different step in every
    environment, some never): the unconstrained ENVP = 1 kernel hands them over to the constrained one."""
    import fastpath_cases
    n_envs, n_steps = 70, 16
    spec, model, qpos0, qvel0, ctrl = fastpath_cases.hand_over_case('salamander_swim', n_envs)
    case, values, physics = run_act_batch(cuda_library, spec, n_envs, n_steps, case=(qpos0, qvel0, ctrl))
    pending = physics.last_pending
    assert 0 < pending < n_envs, pending
    envs = (0, 1, n_envs//2, n_envs - 2, n_envs - 1)
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps)
    print('hand-over', pending, {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < 5e-5, (key, val, worst)


@pytest.mark.gpu
def test_gpu_forcerange_and_wave_rebuild(cuda_library):
    """fb_set_actuator_forcerange and fb_set_wave_controller after the tables are set, on the device."""
    n_envs, n_steps = 64, 10
    spec = spec_of('salamander_swim')
    acts = []

    def setup(p):
        acts.extend(p.model.actuator_id(f'actuator_{k}_{j}') for j in spec.joints_names[:4]
                    for k in ('position', 'velocity'))
    case, values, physics = run_act_batch(cuda_library, spec, n_envs, n_steps, wave=True, setup=setup)
    model, qpos0, qvel0, ctrl, w = case
    physics.set_actuator_forcerange(acts, [1]*len(acts), [[0.0, 0.0]]*len(acts))
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, SAMPLE + (n_envs - 1,), n_steps, wave=w)
    print('switched off', {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < 2e-5, (key, val, worst)


def homogeneous_act_physics(library, spec, model, values, env, n_envs, n_steps):
    """A batch of the model edited to environment env's gains and biases (no table)."""
    from farms_mujoco_b200.engine import BatchedPhysics
    m, _ = edited_act(model, None, values, env)
    physics = BatchedPhysics(m, n_envs, spec.links_names, spec.joints_names, spec.contacts_names, spec.xfrc_names,
                             animat_options=spec.animat_options, arena_options=spec.arena_options,
                             units=spec.simulation_options.units, buffer_size=n_steps + 1, library=library)
    got = physics.env_params()
    for key, val in values.items():
        assert np.array_equal(got[key][0], val[env]), key
    return physics


@pytest.mark.gpu
@pytest.mark.parametrize('name,path,n_envs,slim,wave', [
    ('salamander_swim', 'fast', 64, 0, True),        # SPLIT variant, LEAN + wave
    ('salamander_swim', 'fast', 8192, 7, True),      # SLIM + MULTI
    ('salamander', 'fast', 64, 0, False),            # constrained kernel
    ('salamander_swim', 'team', 64, 0, False),
    ('salamander', 'team', 64, 0, False),            # team kernel on the ground
    ('swimmer8_features', 'fast', 64, 0, False),     # actuation_generic
])
def test_gpu_mixed_batch_equals_homogeneous_batches(cuda_library, name, path, n_envs, slim, wave, monkeypatch):
    """Environment e of a batch with gain and bias tables (the ENVP = 1 kernels) against a batch of
    the model edited to e's values (the default entry points), same kernel variant, same inputs in
    every environment: the same bits, except on the SLIM MULTI layout, where ptxas contracts the
    ENVP = 1 kernel's arithmetic differently (a few ulp, as for the other tables)."""
    from farms_mujoco_b200 import mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    if slim:
        monkeypatch.setenv('FARMS_B200_FAST_BLOCK', '32')        # SLIM needs full warps
    n_steps = 8
    spec = spec_of(name)
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    rng = np.random.default_rng(1)
    qpos0 = np.tile(model.key_qpos, (n_envs, 1))
    qpos0[:, 7:] += rng.uniform(-0.1, 0.1, size=model.nq - 7)
    qvel0 = np.tile(model.key_qvel, (n_envs, 1)) + rng.uniform(-0.3, 0.3, size=model.nv)
    ctrl = np.tile(rng.uniform(-0.3, 0.3, size=model.nu), (n_envs, 1))

    def run(physics):
        physics.set_fast_path(path != 'team')
        if slim:
            physics.set_fast_slim(slim)
        if wave:
            physics.set_wave_controller(*wave_of(spec, model))
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(n_steps)
        return physics.qpos, physics.qvel, physics.log_arrays()

    mixed = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=cuda_library)
    values = act_values(model, n_envs)
    mixed.set_env_params(**values)
    mq, mv, mlogs = run(mixed)
    identical, worst = True, 0.0
    for env in (0, 5, n_envs - 1):
        hq, hv, hlogs = run(homogeneous_act_physics(cuda_library, spec, model, values, env, n_envs, n_steps))
        pairs = [(mq[env], hq[env]), (mv[env], hv[env])] + [(mlogs[k][env], hlogs[k][env]) for k in mlogs]
        for a, b in pairs:
            identical &= np.array_equal(a, b)
            if a.size:
                worst = max(worst, float(np.abs(a.astype(np.float64) - b).max()/max(1e-30, np.abs(b).max())))
    print(name, path, n_envs, 'bit-identical' if identical else f'differs by {worst:.1e} (relative)')
    if slim == 7:
        assert worst < 1e-5, worst
    else:
        assert identical, worst


@pytest.mark.gpu
def test_gpu_full_batch_gains_and_biases(cuda_library):
    """65,536 SALAMANDERs in water with the travelling wave (bench.py's headline configuration) and
    both tables set: 20 launches of 16 steps, no flags, sampled environments close to the oracle on
    their edited models over the first launch."""
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.sharding import synthetic_inputs
    from farms_mujoco_b200 import mjcf_subset
    n_envs, n_steps = 65536, 16
    spec = spec_of('salamander_swim')
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    qpos0, qvel0, _ = synthetic_inputs(model, np.arange(n_envs))
    ctrl = np.zeros((n_envs, model.nu))
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=cuda_library)
    values = act_values(model, n_envs)
    physics.set_env_params(**values)
    w = wave_of(spec, model)
    physics.set_wave_controller(*w)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    assert physics.fast_slim == 7
    physics.step(n_steps)
    assert not physics.flags.any() and physics.last_pending == 0
    sample = (0, 31, 32, 223, 224, n_envs//2, n_envs - 1)
    worst = oracle_act_parity(spec, model, physics, values, qpos0, qvel0, ctrl, sample, n_steps, wave=w)
    print('65536 envs, gains and biases:', {k: f'{v:.1e}' for k, v in worst.items() if v > 0})
    for key, val in worst.items():
        assert val < 5e-5, (key, val, worst)
    for _ in range(19):
        physics.step(n_steps)
    assert not physics.flags.any()
