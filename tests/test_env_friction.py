"""Per-environment contact friction (BatchedPhysics.set_env_params(geom_friction=...), the C ABI's
FB_ENV_CAND_FRICTION).

Environment e of a batch with a friction table must step as the fp64 oracle on the model whose
geoms' sliding frictions are e's row, with the candidates' friction mixed by the compiler's rule
(mjcf_subset.candidate_friction).  The emulation tests run the device code on the host
(conftest.emu_library); the ``-m gpu`` tests run the checks on every constrained kernel variant of
a B200, the hand-over in the middle of a launch, and the comparison with homogeneous batches.
"""

import copy
import dataclasses
import xml.etree.ElementTree as ET

import numpy as np
import pytest

from conftest import make_case, oracle_rollout, parity_errors


def geom_frictions(model, n_envs, seed=11, lo=0.3, hi=2.0):
    """A sliding friction per geom and environment, uniform in [lo, hi]."""
    return np.random.default_rng(seed).uniform(lo, hi, size=(n_envs, model.ngeom))


def joint_values(model, n_envs, seed=7):
    """Per-environment stiffness on every hinge and scaled damping (the free joint keeps 0)."""
    rng = np.random.default_rng(seed)
    hinge = np.asarray(model.jnt_type) != 0
    dof_free = np.asarray(model.jnt_type)[np.asarray(model.dof_jntid)] == 0
    return {'jnt_stiffness': np.where(hinge, rng.uniform(0.005, 0.05, size=(n_envs, model.njnt)), 0.0),
            'dof_damping': np.where(dof_free, 0.0, np.asarray(model.dof_damping)*rng.uniform(0.2, 4.0, size=(n_envs, model.nv)))}


def edited(model, values, env):
    """A copy of model with environment env's values written in: geom_friction[:, 0] and the
    candidates' mixed friction, stiffness, damping."""
    from farms_mujoco_b200.mjcf_subset import candidate_friction
    m = copy.deepcopy(model)
    if 'geom_friction' in values:
        m.geom_friction = np.array(model.geom_friction, dtype=np.float64)
        m.geom_friction[:, 0] = values['geom_friction'][env]
        m.cand_friction = candidate_friction(model, values['geom_friction'][env])
    if 'jnt_stiffness' in values:
        m.jnt_stiffness = np.array(values['jnt_stiffness'][env], dtype=np.float64)
    if 'dof_damping' in values:
        m.dof_damping = np.array(values['dof_damping'][env], dtype=np.float64)
    return m


def mjcf_with_frictions(mjcf, model, frictions, priority=None):
    """The MJCF text with the sliding friction of every collision geom of `model` (and, given, its
    priority) written into the geom's attributes."""
    root = ET.fromstring(mjcf)
    done = set()
    for elem in root.iter('geom'):
        name = elem.get('name')
        if name not in model.geom_names or name in done:
            continue
        g = model.geom_names.index(name)
        rest = ' '.join(repr(float(v)) for v in np.asarray(model.geom_friction)[g, 1:])
        elem.set('friction', f'{float(frictions[g])!r} {rest}')
        if priority is not None:
            elem.set('priority', str(int(priority[g])))
        done.add(name)
    assert len(done) == model.ngeom, (len(done), model.ngeom)
    return ET.tostring(root, encoding='unicode')


def oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps, soft_pairs=False):
    """Worst parity error of each array over `envs`, each against the oracle on its edited model."""
    from farms_mujoco_b200.mjcf_subset import soft_pair_model
    qpos, qvel, logs = physics.qpos, physics.qvel, physics.log_arrays()
    assert not (physics.flags[list(envs)] & 3).any(), physics.flags
    worst = {}
    for env in envs:
        m = edited(model, values, env)
        if soft_pairs:
            m = soft_pair_model(m)
        _, data, states = oracle_rollout(spec, m, physics.tables, n_steps + 1, qpos0[env], qvel0[env], ctrl[env])
        errs = parity_errors(qpos[env], qvel[env], {k: v[env] for k, v in logs.items()}, *states[-1], data)
        errs.pop('detail')
        for key, val in errs.items():
            worst[key] = max(worst.get(key, 0.0), val)
    return worst


def spec_of(name):
    import variant_models
    from farms_mujoco_b200 import models
    if name == 'salamander_box_feet':
        return variant_models.salamander_box_feet()
    if name == 'salamander_foot_pairs':
        return variant_models.salamander_foot_pairs(swimming=False)
    return models.MODELS[name]()


def inputs(name, n_envs, seed=0):
    """make_case's seeded inputs for `name` (foot pairs: legs folded so that the feet touch)."""
    from farms_mujoco_b200 import mjcf_subset
    spec = spec_of(name)
    if name in ('salamander', 'centipede'):
        return make_case(name, n_envs, seed=seed)
    import variant_models
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    rng = np.random.default_rng(seed)
    key = variant_models.folded_legs_qpos(model, 1.0) if name == 'salamander_foot_pairs' else model.key_qpos
    qpos0 = np.tile(key, (n_envs, 1))
    qpos0[:, 7:] += rng.uniform(-0.03, 0.03, size=(n_envs, model.nq - 7))
    qvel0 = rng.uniform(-0.2, 0.2, size=(n_envs, model.nv))
    ctrl = rng.uniform(-0.3, 0.3, size=(n_envs, model.nu))
    return spec, model, qpos0, qvel0, ctrl


def run_batch(library, name, n_envs, n_steps, path='fast', joints=False, setup=None, case=None):
    """One batch with per-environment geom frictions (and, with `joints`, stiffness and damping)
    stepped n_steps on one kernel path: 'fast' (per-thread kernels), 'fast_team' (team kernel on the
    hand-overs) or 'team'.  Returns the case, the values and the batch."""
    from farms_mujoco_b200.engine import BatchedPhysics
    spec, model, qpos0, qvel0, ctrl = case or inputs(name, n_envs)
    physics = BatchedPhysics(model, n_envs, spec.links_names, spec.joints_names, spec.contacts_names,
                             spec.xfrc_names, animat_options=spec.animat_options, arena_options=spec.arena_options,
                             units=spec.simulation_options.units, buffer_size=n_steps + 1, library=library)
    if path == 'team':
        physics.set_fast_path(False)
    elif path == 'fast_team':
        physics.set_constraint_path(False)
    if setup:
        setup(physics)
    values = {'geom_friction': geom_frictions(model, n_envs)}
    if joints:
        values.update(joint_values(model, n_envs))
    physics.set_env_params(**values)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    return (spec, model, qpos0, qvel0, ctrl), values, physics


# ----------------------------------------------------------------------------------- API
def test_api_validation_and_read_back(emu_library):
    from farms_mujoco_b200.engine import BatchedPhysics, EngineError
    from farms_mujoco_b200.mjcf_subset import candidate_friction
    spec, model, qpos0, qvel0, _ = make_case('salamander', 3)
    physics = BatchedPhysics.from_spec(spec, 3, buffer_size=2, library=emu_library)
    base = np.asarray(model.geom_friction)[:, 0]
    got = physics.env_params()['geom_friction']
    assert got.shape == (3, model.ngeom) and np.array_equal(got, np.tile(base, (3, 1)))
    lib, h = physics.lib, physics._handle       # pylint: disable=protected-access

    def cand_table():
        out = np.zeros((3, model.ncand))
        assert lib.fb_get_env_param(h, 4, out.ctypes.data_as(ct_double_p())) == 0
        return out

    assert np.array_equal(cand_table(), np.tile(model.cand_friction, (3, 1)))

    G = geom_frictions(model, 3)
    # refusals in Python: negative or non-finite geom values, named by environment and geom
    for bad_value, match in ((-0.5, 'is -0.5'), (np.nan, 'is nan'), (np.inf, 'is inf')):
        bad = G.copy()
        bad[2, 4] = bad_value
        with pytest.raises(ValueError, match=rf'environment 2, geom 4 \("{model.geom_names[4]}"\) {match}'):
            physics.set_env_params(geom_friction=bad)
    # a mixed value below 0.1: the engine's refusal, re-worded with the two geoms of the candidate
    bad = G.copy()
    g2 = int(model.cand_geom2[5])
    bad[1, :] = np.where(np.arange(model.ngeom) == g2, 0.05, bad[1, :])
    bad[1, model.cand_geom1[5]] = 0.0                       # the plane: the max rule takes the foot's
    first = int(np.argmax(candidate_friction(model, bad[1]) < 0.1))
    names = model.geom_names[model.cand_geom1[first]], model.geom_names[model.cand_geom2[first]]
    with pytest.raises(EngineError, match=rf'environment 1 mixes to 0.05 on candidate {first}, geoms "{names[0]}" and '
                                          rf'"{names[1]}".*FB_ENV_CAND_FRICTION.*below 0.1 at environment 1, '
                                          rf'candidate {first}.*1/mu\^2'):
        physics.set_env_params(geom_friction=bad)
    with pytest.raises(ValueError, match='geom_friction'):
        physics.set_env_params(geom_friction=np.ones(model.ngeom + 1))
    # the engine's own refusals, by candidate: non-finite, below the floor
    for value, match in ((np.nan, 'non-finite value at environment 0, candidate 3'),
                         (0.09, 'below 0.1 at environment 0, candidate 3')):
        table = np.tile(model.cand_friction, (3, 1))
        table[0, 3] = value
        assert lib.fb_set_env_param(h, 4, table.ctypes.data_as(ct_double_p())) != 0
        assert match in lib.fb_last_error().decode()
    # nothing of the refused calls was kept
    assert np.array_equal(physics.env_params()['geom_friction'], np.tile(base, (3, 1)))
    assert np.array_equal(cand_table(), np.tile(model.cand_friction, (3, 1)))

    # broadcasting, read-back, the candidates' table
    physics.set_env_params(geom_friction=G[0])
    assert np.array_equal(physics.env_params()['geom_friction'], np.tile(G[0], (3, 1)))
    assert np.array_equal(cand_table(), np.tile(candidate_friction(model, G[0]), (3, 1)))
    physics.set_env_params(geom_friction=G)
    assert np.array_equal(physics.env_params()['geom_friction'], G)
    assert np.array_equal(cand_table(), candidate_friction(model, G))
    # only the keywords passed change; the table survives reset
    physics.set_env_params(dof_damping=np.asarray(model.dof_damping)*2)
    physics.reset(qpos0, qvel0)
    assert np.array_equal(physics.env_params()['geom_friction'], G)
    assert np.array_equal(cand_table(), candidate_friction(model, G))
    # None: the model's value again
    physics.set_env_params(geom_friction=None)
    assert np.array_equal(physics.env_params()['geom_friction'], np.tile(base, (3, 1)))
    assert np.array_equal(cand_table(), np.tile(model.cand_friction, (3, 1)))
    physics.close()


def ct_double_p():
    from farms_mujoco_b200 import cabi
    return cabi.c_double_p


def test_pair_candidates_keep_the_model_value(emu_library):
    """An explicit <pair> takes its friction from the pair element: the engine refuses a table that
    changes it, and candidate_friction leaves it as compiled."""
    import variant_models
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.mjcf_subset import candidate_friction
    spec = variant_models.salamander_foot_pairs(swimming=False)
    physics = BatchedPhysics.from_spec(spec, 2, buffer_size=2, library=emu_library)
    model = physics.model
    pair = np.flatnonzero(np.isin(model.cand_end, (20, 21)))
    assert len(pair) == 2
    mixed = candidate_friction(model, geom_frictions(model, 2))
    assert np.array_equal(mixed[:, pair], np.tile(model.cand_friction[pair], (2, 1)))
    table = np.ascontiguousarray(mixed)
    table[1, pair[1]] = 0.8
    assert physics.lib.fb_set_env_param(physics._handle, 4, table.ctypes.data_as(ct_double_p())) != 0  # pylint: disable=protected-access
    err = physics.lib.fb_last_error().decode()
    assert f'differs from the <pair> candidate\'s friction' in err and f'environment 1, candidate {pair[1]}' in err, err
    physics.set_env_params(geom_friction=geom_frictions(model, 2))
    physics.close()


# ------------------------------------------------------------------ mixing rule = the compiler's
@pytest.mark.parametrize('name,priority', [('salamander', False), ('salamander_box_feet', False),
                                           ('salamander', True), ('salamander_foot_pairs', False)])
def test_candidate_friction_matches_the_compiler(name, priority):
    """candidate_friction of random per-geom frictions equals what parse_mjcf compiles from the MJCF
    with those frictions written into the geoms."""
    from farms_mujoco_b200.mjcf_subset import candidate_friction, parse_mjcf
    spec = spec_of(name)
    model = parse_mjcf(spec.mjcf)
    rng = np.random.default_rng(3)
    if name == 'salamander_box_feet':
        assert np.bincount(model.cand_geom2).max() == 8            # eight corners per box
    prio = None
    if priority:
        # unequal priorities: the higher one's friction, whichever is larger
        prio = rng.integers(0, 3, size=model.ngeom)
        model.geom_priority = prio.astype(np.int32)
        assert (prio[model.cand_geom1] != prio[model.cand_geom2]).any()
    for seed in range(3):
        G = np.random.default_rng(seed).uniform(0.0, 2.0, size=model.ngeom)
        G[np.random.default_rng(seed).integers(0, model.ngeom)] = 0.0     # a frictionless geom: the floor
        ref = parse_mjcf(mjcf_with_frictions(spec.mjcf, model, G, prio))
        assert np.array_equal(candidate_friction(model, G), ref.cand_friction), seed
        assert np.array_equal(candidate_friction(model, np.stack([G, G[::-1]]))[0], ref.cand_friction)
    if name == 'salamander_foot_pairs':
        pair = np.isin(model.cand_end, (20, 21))
        assert pair.any() and np.array_equal(candidate_friction(model, G)[pair], model.cand_friction[pair])


# ------------------------------------------------------------------------------ clearing
def test_cleared_table_is_bit_identical(emu_library):
    """A friction table set and then cleared leaves the default path: the same bits as a batch that
    never set one."""
    from farms_mujoco_b200.engine import BatchedPhysics
    spec, model, qpos0, qvel0, ctrl = make_case('salamander', 3)
    out = []
    for clear in (False, True):
        physics = BatchedPhysics.from_spec(spec, 3, buffer_size=5, library=emu_library)
        if clear:
            physics.set_env_params(geom_friction=geom_frictions(model, 3))
            physics.set_env_params(geom_friction=None)
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(4)
        assert physics.last_pending == 3
        out.append((physics.qpos, physics.log_arrays()))
    assert np.array_equal(out[0][0], out[1][0])
    for kind in out[0][1]:
        assert np.array_equal(out[0][1][kind], out[1][1][kind]), kind


# -------------------------------------------------------------------- oracle parity (host)
@pytest.mark.parametrize('name,path,joints,n_steps,tol', [
    ('salamander', 'fast', False, 8, 2e-5),           # per-thread constrained kernel (fastc)
    ('centipede', 'fast', False, 6, 1e-4),
    ('salamander', 'team', False, 8, 5e-3),           # team kernel
    ('salamander_box_feet', 'fast', False, 6, 1e-4),
    ('salamander', 'fast', True, 8, 2e-5),            # friction, stiffness and damping together
])
def test_oracle_parity_emulated(emu_library, name, path, joints, n_steps, tol):
    case, values, physics = run_batch(emu_library, name, 4, n_steps, path=path, joints=joints)
    spec, model, qpos0, qvel0, ctrl = case
    if path == 'fast':
        assert physics.last_pending == 4                # the constrained kernel stepped them
    assert np.abs(physics.log_arrays()['contacts']).max() > 0
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, range(4), n_steps)
    print(name, path, 'joints' if joints else '', {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < (max(5e-4, tol) if key == 'contacts' else tol), (key, val, worst)


def test_oracle_parity_foot_pairs_team_emulated(emu_library):
    """Foot pairs (two-body rows: team kernel only) with per-environment plane frictions beside the
    pairs' own mu = 0.5: the pairs' rows go through the same access and keep the pair's value."""
    n_envs, n_steps = 3, 6
    case, values, physics = run_batch(emu_library, 'salamander_foot_pairs', n_envs, n_steps)
    spec, model, qpos0, qvel0, ctrl = case
    assert physics.fast_path == 0
    pair = np.isin(model.cand_end, (20, 21))
    assert np.all(model.cand_friction[pair] == 0.5)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, range(n_envs), n_steps)
    print('foot pairs team', {k: f'{v:.2e}' for k, v in worst.items()})
    for key, val in worst.items():
        assert val < 5e-3, (key, val, worst)


# ------------------------------------------------------------ physics without the oracle
def test_contact_forces_lie_in_each_environments_pyramid(emu_library):
    """The contact forces of every environment (team kernel's derived view: normal, t1, t2 per
    contact) satisfy |f_t1| + |f_t2| <= mu_e f_n with that environment's mixed mu: a write-back with
    another environment's mu, or the model's, leaves the pyramid."""
    from farms_mujoco_b200.engine import BatchedPhysics
    n_envs = 4
    spec, model, qpos0, qvel0, ctrl = make_case('salamander', n_envs)
    qvel0[:, 0] += 0.3                                           # sliding forward
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=8, library=emu_library)
    mu = np.array([0.3, 0.6, 1.2, 2.0])
    physics.set_env_params(geom_friction=np.repeat(mu[:, None], model.ngeom, axis=1))
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    ratios = []
    for _ in range(4):
        physics.step(1, want_derived=True)
        d = physics.derived()
        for e in range(n_envs):
            n = int(d['ncon'][e])
            if n == 0:
                continue
            f = d['con_force'][e, :n].astype(np.float64)
            assert (f[:, 0] >= 0).all()
            r = (np.abs(f[:, 1]) + np.abs(f[:, 2]))/np.maximum(f[:, 0], 1e-30)
            assert (np.abs(f[:, 1]) + np.abs(f[:, 2]) <= mu[e]*f[:, 0]*(1 + 1e-5) + 1e-9).all(), (e, r.max(), mu[e])
            ratios.append((e, r.max()/mu[e]))
    print('max tangential / (mu_e normal) per environment and step:', [f'{e}:{v:.3f}' for e, v in ratios])
    # a sliding contact's force is on the edge of its own environment's pyramid: in the mu = 0.3 and
    # 0.6 environments the largest ratio reaches that environment's mu (a mu of another environment,
    # or the model's mu = 1, would put it at 0.3 / 0.6 of it, or over the bound above)
    for e in (0, 1):
        assert max(v for k, v in ratios if k == e) > 0.95, (e, mu[e], ratios)
    physics.close()


def test_slide_distance_decreases_with_friction(emu_library):
    """The same body pushed sideways over the ground, one mu per environment: the slide is strictly
    shorter where the friction is larger."""
    from farms_mujoco_b200.engine import BatchedPhysics
    n_envs, n_steps = 5, 150
    spec, model, qpos0, qvel0, ctrl = make_case('salamander', 1, qvel_scale=0.0, ctrl_scale=0.0)
    qpos0, qvel0, ctrl = (np.repeat(a, n_envs, axis=0) for a in (qpos0, qvel0, ctrl))
    qvel0[:, 1] = 0.3                                            # sideways, 0.3 m/s
    # frictions low enough that the body slides rather than tips over its feet (from mu ~ 1 up, the
    # legs catch and the body rolls, and the distance no longer follows mu)
    mu = np.array([0.1, 0.2, 0.3, 0.45, 0.6])
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=2, library=emu_library)
    physics.set_env_params(geom_friction=np.repeat(mu[:, None], model.ngeom, axis=1))
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(n_steps)
    assert not physics.flags.any()
    slide = physics.qpos[:, 1] - qpos0[:, 1]
    print('mu', mu, 'slide [mm]', np.round(1e3*slide, 3))
    assert (slide > 0).all() and (np.diff(slide) < 0).all(), slide


# ----------------------------------------------------------------------------------- B200
SAMPLE = (0, 1, 31, 32, 33)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['salamander', 'centipede'])
@pytest.mark.parametrize('blk', [16, 32])
@pytest.mark.parametrize('lean', [True, False])
@pytest.mark.parametrize('split', [True, False])
def test_gpu_oracle_parity_constrained(cuda_library, name, blk, lean, split, monkeypatch):
    """Every variant of the per-thread constrained kernel with ENVP = 1: BLK 16 / 32, LEAN and
    general, the SPLIT constrained kernel on and off."""
    monkeypatch.setenv('FARMS_B200_FAST_BLOCK', str(blk))
    n_envs, n_steps = 64, 8

    def setup(p):
        p.set_fast_lean(lean)
        p.set_con_split(split)
    case, values, physics = run_batch(cuda_library, name, n_envs, n_steps, setup=setup)
    spec, model, qpos0, qvel0, ctrl = case
    assert physics.fast_path and physics.last_pending == n_envs and physics.con_split == split
    print(name, 'blk', blk, 'lean' if lean else 'general', 'con_split', physics.con_split)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, SAMPLE + (n_envs - 1,), n_steps)
    print({k: f'{v:.2e}' for k, v in worst.items()})
    tol = 2e-5 if name == 'salamander' else 1e-4
    physics.close()
    for key, val in worst.items():
        assert val < (5e-4 if key == 'contacts' else tol), (key, val, worst)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['salamander', 'centipede'])
@pytest.mark.parametrize('path', ['fast_team', 'team'])
def test_gpu_oracle_parity_team(cuda_library, name, path):
    n_envs, n_steps = 64, 8
    case, values, physics = run_batch(cuda_library, name, n_envs, n_steps, path=path)
    spec, model, qpos0, qvel0, ctrl = case
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, SAMPLE + (n_envs - 1,), n_steps)
    print(name, path, {k: f'{v:.2e}' for k, v in worst.items()})
    physics.close()
    for key, val in worst.items():
        assert val < (5e-3 if key == 'contacts' else 5e-4), (key, val, worst)


def touch_down_case(n_envs, seed=5):
    """Ground batch whose environments start above the ground at different heights, falling at
    4 m/s: the higher ones enter the per-thread kernel's conservative plane bound (about 6 cm) after
    a few steps, and they touch down at different steps of one 16-step launch.  The first starts on
    the ground, the last never comes near it."""
    spec, model, qpos0, qvel0, ctrl = make_case('salamander', n_envs, qvel_scale=0.05)
    lift = np.random.default_rng(seed).uniform(0.02, 0.09, size=n_envs)
    lift[0], lift[-1] = 0.0, 0.2
    qpos0[:, 2] += lift
    qvel0[:, 2] = np.where(lift > 0, -4.0, qvel0[:, 2])
    return spec, model, qpos0, qvel0, ctrl


@pytest.mark.gpu
def test_gpu_touch_down_mid_launch(cuda_library):
    """A friction table alone: the unconstrained default kernel steps the falling environments and
    hands each over to the constrained ENVP = 1 kernel at its touch-down step, in the middle of one launch."""
    n_envs, n_steps = 70, 16
    case = touch_down_case(n_envs)
    _, values, physics = run_batch(cuda_library, 'salamander', n_envs, n_steps, case=case)
    spec, model, qpos0, qvel0, ctrl = case
    pending = physics.last_pending
    assert 1 < pending < n_envs, pending
    contacts = np.abs(physics.log_arrays()['contacts']).sum(axis=(2, 3))      # [env, row]
    first = [int(np.argmax(c > 0)) if (c > 0).any() else -1 for c in contacts]
    assert len({f for f in first if f > 1}) > 3, first                     # touch-downs spread over the launch
    # fewer environments are inside the plane bound at the first step: the others were handed over
    # in the middle of the launch
    first_step = run_batch(cuda_library, 'salamander', n_envs, 1, case=case)[2]
    assert first_step.last_pending < pending, (first_step.last_pending, pending)
    first_step.close()
    envs = (0, 1, 2, n_envs//2, n_envs - 2, n_envs - 1)
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps)
    print('touch-down', pending, 'first contact rows', sorted(set(first)), {k: f'{v:.2e}' for k, v in worst.items()})
    physics.close()
    for key, val in worst.items():
        assert val < (5e-4 if key == 'contacts' else 5e-5), (key, val, worst)


def homogeneous_physics(library, spec, model, G, env, n_envs, n_steps):
    """A batch of the MJCF edited to environment env's geom frictions (no table): the default entry
    points."""
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.mjcf_subset import parse_mjcf
    spec = dataclasses.replace(spec, mjcf=mjcf_with_frictions(spec.mjcf, model, G[env]))
    m = parse_mjcf(spec.mjcf)
    physics = BatchedPhysics(m, n_envs, spec.links_names, spec.joints_names, spec.contacts_names, spec.xfrc_names,
                             animat_options=spec.animat_options, arena_options=spec.arena_options,
                             units=spec.simulation_options.units, buffer_size=n_steps + 1, library=library)
    assert np.array_equal(physics.env_params()['geom_friction'][0], G[env])
    return physics


@pytest.mark.gpu
@pytest.mark.parametrize('name,path', [('salamander', 'fast'), ('centipede', 'fast'), ('salamander', 'team')])
def test_gpu_mixed_batch_equals_homogeneous_batches(cuda_library, name, path):
    """Environment e of a batch with a friction table (the constrained ENVP = 1 kernel, or the team kernel
    reading the table) against a batch of the MJCF edited to e's frictions (the default entry
    points), same inputs in every environment: bit-identical, or within 1e-5 relative where ptxas
    contracts the ENVP = 1 kernels differently."""
    from farms_mujoco_b200.engine import BatchedPhysics
    n_envs, n_steps = 64, 8
    spec, model, qpos0, qvel0, ctrl = make_case(name, 1)
    qpos0, qvel0, ctrl = (np.repeat(a, n_envs, axis=0) for a in (qpos0, qvel0, ctrl))

    def run(physics):
        physics.set_fast_path(path != 'team')
        physics.reset(qpos0, qvel0)
        physics.set_ctrl(ctrl)
        physics.step(n_steps)
        out = physics.qpos, physics.qvel, physics.log_arrays()
        physics.close()
        return out

    mixed = BatchedPhysics.from_spec(spec, n_envs, buffer_size=n_steps + 1, library=cuda_library)
    G = geom_frictions(model, n_envs)
    mixed.set_env_params(geom_friction=G)
    mq, mv, mlogs = run(mixed)
    identical, worst = True, 0.0
    for env in (0, 5, 32, n_envs - 1):
        hq, hv, hlogs = run(homogeneous_physics(cuda_library, spec, model, G, env, n_envs, n_steps))
        pairs = [(mq[env], hq[env]), (mv[env], hv[env])] + [(mlogs[k][env], hlogs[k][env]) for k in mlogs]
        for a, b in pairs:
            identical &= np.array_equal(a, b)
            if a.size:
                worst = max(worst, float(np.abs(a.astype(np.float64) - b).max()/max(1e-30, np.abs(b).max())))
    print(name, path, n_envs, 'bit-identical' if identical else f'differs by {worst:.1e} (relative)')
    assert worst < 1e-5, worst


@pytest.mark.gpu
@pytest.mark.parametrize('name,n_envs', [('salamander', 4096), ('centipede', 8192)])
def test_gpu_scale_friction_stiffness_damping(cuda_library, name, n_envs):
    """4,096 SALAMANDERs / 8,192 CENTIPEDEs on the ground, 16 steps in one launch, with friction,
    stiffness and damping set: no flags, sampled environments within tolerance of the oracle."""
    n_steps = 16
    case, values, physics = run_batch(cuda_library, name, n_envs, n_steps, joints=True)
    spec, model, qpos0, qvel0, ctrl = case
    assert not physics.flags.any() and physics.last_pending == n_envs
    rng = np.random.default_rng(3)
    envs = sorted({0, 31, 32, n_envs//2, n_envs - 1} | set(int(e) for e in rng.integers(0, n_envs, size=3)))
    worst = oracle_parity(spec, model, physics, values, qpos0, qvel0, ctrl, envs, n_steps)
    print(name, n_envs, {k: f'{v:.2e}' for k, v in worst.items()})
    tol = 5e-5 if name == 'salamander' else 2e-4
    physics.close()
    for key, val in worst.items():
        assert val < (1e-3 if key == 'contacts' else tol), (key, val, worst)
