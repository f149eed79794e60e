"""Per-environment episodes: restart some environments of a batch while the others keep running
(fb_reset_envs, fb_reset_envs_where, BatchedPhysics.reset_envs).

A restarted environment e must step as environment e of a freshly reset batch given its restart
state (the episode clock gives the travelling-wave controller the episode's time), and its log
accessors must return that episode; the other environments must step as in a batch that was never
restarted.  The emulation tests run the device code on the host (conftest.emu_library); the ``-m
gpu`` tests run the same comparisons on every kernel path of a B200, the device-mask entry point,
pipelined host calls and a full-size batch.
"""

import numpy as np
import pytest

from conftest import make_case, parity_errors

KINDS = ('links', 'joints', 'contacts', 'xfrc')


def wave_physics(library, spec, model, n_envs, ring, phase, log_stride=1, setup=None):
    """A batch with the on-device travelling-wave controller (the one step code that reads time)."""
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.models import travelling_wave_parameters
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=ring, library=library, log_stride=log_stride)
    if setup:
        setup(physics)
    joints, amp, freq, lag = travelling_wave_parameters(spec)
    physics.set_env_phase(phase)
    physics.set_wave_controller([model.actuator_id(f'actuator_position_{j}') for j in joints], amp, freq, lag)
    return physics


def wave_controller(spec, model, phase):
    """The oracle's controller for the wave of wave_physics: time is the rollout's own (episode) time."""
    from farms_mujoco_b200.models import travelling_wave_parameters
    joints, amp, freq, lag = travelling_wave_parameters(spec)
    acts = [model.actuator_id(f'actuator_position_{j}') for j in joints]

    def controller(iteration, time):
        ctrl = np.zeros(model.nu)
        ctrl[acts] = amp*np.sin(2*np.pi*freq*time - lag + phase)
        return ctrl
    return controller


def restart_states(model, qpos0, qvel0, envs, seed=9):
    """New states for the restarted environments: even entries given rows, odd ones the keyframe."""
    rng = np.random.default_rng(seed)
    q = np.tile(model.key_qpos, (len(envs), 1))
    q[:, 7:] += rng.uniform(-0.1, 0.1, size=(len(envs), model.nq - 7))
    v = np.tile(model.key_qvel, (len(envs), 1)) + rng.uniform(-0.2, 0.2, size=(len(envs), model.nv))
    keyframe = np.arange(len(envs)) % 2 == 1
    q[keyframe], v[keyframe] = model.key_qpos, model.key_qvel
    return q, v, keyframe


class Scenario:
    """Batch A: reset, K1 steps, restart `envs`, K2 steps.  B: never restarted, K1 + K2 steps.
    C: fresh, reset to A's restart states in the restarted environments, K2 steps."""

    def __init__(self, library, name, n_envs, envs, k1, k2, ring, log_stride=1, setup=None, chunks=None,
                 keyframe_call=True):
        spec, model, qpos0, qvel0, _ = make_case(name, n_envs)
        self.spec, self.model, self.envs, self.k2 = spec, model, list(envs), k2
        self.phase = np.random.default_rng(2).uniform(0, 2*np.pi, n_envs)
        make = lambda: wave_physics(library, spec, model, n_envs, ring, self.phase, log_stride, setup)
        q, v, keyframe = restart_states(model, qpos0, qvel0, self.envs)
        self.start_q, self.start_v = qpos0.copy(), qvel0.copy()
        self.start_q[self.envs], self.start_v[self.envs] = q, v
        self.A, self.B, self.C = make(), make(), make()
        self.A.reset(qpos0, qvel0)
        self.B.reset(qpos0, qvel0)
        self.C.reset(self.start_q, self.start_v)
        for physics in (self.A, self.B):
            physics.step(k1*log_stride)
        self.it = self.A.iteration
        given = [e for e, kf in zip(self.envs, keyframe) if not kf]
        kf = [e for e, kf in zip(self.envs, keyframe) if kf]
        if keyframe_call:
            # two calls: the given rows, then the keyframe (NULL rows)
            self.A.reset_envs(given, q[~keyframe], v[~keyframe])
            self.A.reset_envs(kf)
        else:
            self.A.reset_envs(self.envs, q, v)
        for physics in (self.A, self.B, self.C):
            for n in (chunks or [k2]):
                physics.step(n*log_stride)

    def others(self):
        return [e for e in range(self.A.n_envs) if e not in self.envs]


def differences(pairs):
    """(bit-identical, worst relative difference) over (ours, reference) array pairs."""
    identical, worst = True, 0.0
    for a, b in pairs:
        a, b = np.asarray(a), np.asarray(b)
        assert a.shape == b.shape, (a.shape, b.shape)
        identical &= np.array_equal(a, b)
        if a.size:
            worst = max(worst, float(np.abs(a.astype(np.float64) - b).max()/max(1e-30, float(np.abs(b).max()))))
    return identical, worst


def compare(sc, exact=True, tol=1e-6):
    """Restarted environments against the fresh batch C, the others against the never-restarted
    batch B: state, and every log kind through export_farms and log_arrays(env=).  exact: the same
    bits; else (two compilations of the same arithmetic, which ptxas may contract differently)
    `tol` relative."""
    A, B, C = sc.A, sc.B, sc.C
    assert not (A.flags & 1).any()
    qa, va, qb, vb, qc, vc = A.qpos, A.qvel, B.qpos, B.qvel, C.qpos, C.qvel
    pairs_new, pairs_old = [], []
    for e in sc.envs:
        pairs_new += [(qa[e], qc[e]), (va[e], vc[e])]
        xa, xc = A.export_farms(e), C.export_farms(e)
        pairs_new += [(getattr(xa.sensors, k).array, getattr(xc.sensors, k).array) for k in KINDS]
        la, lc = A.log_arrays(env=e), C.log_arrays(env=e)
        pairs_new += [(la[k], lc[k]) for k in KINDS]
        # export_farms and log_arrays(env=) agree
        pairs_new += [(getattr(xa.sensors, k).array, la[k].astype(np.float64)) for k in KINDS]
    la, lb = A.log_arrays(), B.log_arrays()
    for e in sc.others():
        pairs_old += [(qa[e], qb[e]), (va[e], vb[e])] + [(la[k][e], lb[k][e]) for k in KINDS]
    for label, pairs in (('restarted', pairs_new), ('others', pairs_old)):
        identical, worst = differences(pairs)
        print(label, 'bit-identical' if identical else f'differs by {worst:.1e} (relative)')
        if exact:
            assert identical, (label, worst)
        else:
            assert worst < tol, (label, worst)


# ----------------------------------------------------------------------------------- API
def test_api(emu_library):
    from farms_mujoco_b200.engine import BatchedPhysics, EngineError
    spec, model, qpos0, qvel0, ctrl = make_case('salamander_swim', 5)
    physics = BatchedPhysics.from_spec(spec, 5, buffer_size=4, library=emu_library)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(3)
    assert np.array_equal(physics.episode_start(), np.zeros(5, np.int64))
    good_q, good_v = qpos0[:2].copy(), qvel0[:2].copy()
    with pytest.raises(EngineError, match=r'envs\[1\] = 5 is out of range \[0, 5\)'):
        physics.reset_envs([0, 5])
    with pytest.raises(EngineError, match=r'envs\[0\] = -1 is out of range'):
        physics.reset_envs([-1])
    with pytest.raises(EngineError, match=r'environment 3 is given twice \(envs\[0\] and envs\[2\]\)'):
        physics.reset_envs([3, 1, 3])
    bad = good_q.copy()
    bad[1, 9] = np.nan
    with pytest.raises(EngineError, match=r'non-finite qpos0 at row 1 \(environment 4\), index 9'):
        physics.reset_envs([2, 4], bad, good_v)
    bad = good_v.copy()
    bad[0, 2] = np.inf
    with pytest.raises(EngineError, match=r'non-finite qvel0 at row 0 \(environment 2\), index 2'):
        physics.reset_envs([2, 4], good_q, bad)
    with pytest.raises(ValueError, match=r'qpos must be \[2, '):
        physics.reset_envs([2, 4], qpos0)
    lib = physics.lib
    assert lib.fb_reset_envs(None, 0, None, None, None) != 0 and b'null handle' in lib.fb_last_error()
    assert lib.fb_reset_envs_where(physics._handle, None, None, None) != 0
    assert b'null mask' in lib.fb_last_error()
    # refused calls changed nothing; an empty list (or an all-false mask) enqueues nothing
    before = (physics.qpos, physics.qvel, physics.ctrl, physics.log_arrays(), physics.launch_count())
    physics.reset_envs([])
    physics.reset_envs(np.zeros(5, bool))
    after = (physics.qpos, physics.qvel, physics.ctrl, physics.log_arrays(), physics.launch_count())
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    assert np.array_equal(before[2], after[2]) and before[4] == after[4]
    for kind in KINDS:
        assert before[3][kind].tobytes() == after[3][kind].tobytes(), kind
    assert np.array_equal(physics.episode_start(), np.zeros(5, np.int64))
    # a bool mask picks its rows; episode_start reads back; the batch counter stays
    mask = np.array([False, True, False, True, False])
    physics.reset_envs(mask, qpos0, qvel0)
    assert np.array_equal(physics.episode_start(), [0, 3, 0, 3, 0]) and physics.iteration == 3
    iteration = physics._read(physics.state_view.iteration_dev, (5,), np.int64)
    assert np.array_equal(iteration, [3, 3, 3, 3, 3])
    assert np.array_equal(physics.qpos[[1, 3]], qpos0[[1, 3]].astype(np.float32))
    assert not physics.ctrl[[1, 3]].any() and np.array_equal(physics.ctrl[[0, 2, 4]], ctrl[[0, 2, 4]].astype(np.float32))
    physics.step(2)
    physics.reset_envs([1])
    assert np.array_equal(physics.episode_start(), [0, 5, 0, 3, 0])
    assert np.array_equal(physics.qpos[1], model.key_qpos.astype(np.float32))
    physics.reset(qpos0, qvel0)
    assert np.array_equal(physics.episode_start(), np.zeros(5, np.int64))
    with pytest.raises(TypeError, match='integer indices or a bool mask'):
        physics.reset_envs([0.5])
    # between the sub-steps of a logged iteration
    sub = BatchedPhysics.from_spec(spec, 5, buffer_size=4, library=emu_library, log_stride=2)
    sub.reset(qpos0, qvel0)
    sub.step(1)
    with pytest.raises(ValueError, match='not a full step'):
        sub.reset_envs([0])
    sub.step(1)
    sub.reset_envs([0])
    assert sub.episode_start()[0] == 2


# ----------------------------------------------------------------------------- core parity
@pytest.mark.parametrize('name,ring,chunks', [
    ('swimmer8', 16, None),
    ('salamander_swim', 16, None),
    ('salamander_swim', 5, [4, 3, 5]),          # the ring wraps, several launches
    ('salamander', 16, None),                   # ground: the constrained kernel
])
def test_core_parity(emu_library, name, ring, chunks):
    sc = Scenario(emu_library, name, 9, envs=[1, 4, 5, 8], k1=6, k2=12, ring=ring, chunks=chunks)
    assert np.array_equal(sc.A.episode_start()[sc.envs], [6]*4)
    compare(sc)


@pytest.mark.parametrize('name', ['salamander_swim', 'salamander'])
def test_core_parity_split(emu_library, name):
    """SPLIT variants (several warps per environment group; emu_split_run), unconstrained and
    constrained."""
    def setup(physics):
        physics.set_fast_split(True)
        physics.set_con_split(True)
    sc = Scenario(emu_library, name, 6, envs=[0, 3, 5], k1=5, k2=8, ring=16, setup=setup)
    assert sc.A.fast_split > 1
    compare(sc)


def test_core_parity_team(emu_library):
    sc = Scenario(emu_library, 'salamander_swim', 6, envs=[2, 3], k1=5, k2=8, ring=16,
                  setup=lambda p: p.set_fast_path(False), keyframe_call=False)
    compare(sc)


@pytest.mark.parametrize('name', ['salamander_swim', 'salamander'])
def test_against_oracle(emu_library, name):
    """Restarted environments against the fp64 oracle from their restart state, K2 steps, with the
    wave controller's time starting at the restart (tolerances of test_env_params)."""
    from oracle.oracle import OraclePhysics
    from oracle import farms_oracle as fo
    sc = Scenario(emu_library, name, 6, envs=[1, 4], k1=7, k2=10, ring=11)
    qpos, qvel = sc.A.qpos, sc.A.qvel
    for e in sc.envs:
        ctl = wave_controller(sc.spec, sc.model, sc.phase[e])
        data, states = fo.reference_rollout(OraclePhysics(sc.model), sc.spec, sc.A.tables, sc.k2 + 1,
                                            controller=ctl, qpos0=sc.start_q[e], qvel0=sc.start_v[e])
        logs = {k: getattr(sc.A.export_farms(e).sensors, k).array for k in KINDS}
        errs = parity_errors(qpos[e], qvel[e], logs, *states[-1], data)
        errs.pop('detail')
        print(name, e, {k: f'{v:.1e}' for k, v in errs.items()})
        for key, val in errs.items():
            assert val < (5e-4 if key == 'contacts' else 2e-5), (key, val)


def test_cpg_rows_restored(emu_library):
    """On-device CPG with spring references: a restarted environment's oscillators return to the
    state fb_set_cpg_state set (rates 0), and it then steps as in a fresh batch."""
    import fastpath_cases
    from farms_mujoco_b200.engine import BatchedPhysics
    n = 5
    spec, model, qpos0, qvel0, _ = make_case('swimmer8', n)
    spring_joints = ('joint_5', 'joint_6')
    cpg = fastpath_cases.swimmer_cpg(n, True, spring_joints=spring_joints)
    ctrl_names = [model.actuator_names[a] for a in range(model.nu)]
    net = cpg.device_cpg(lambda joint, kind: ctrl_names.index(f'actuator_position_{joint}'),
                         spring_index=lambda joint: int(model.jnt_qposadr[model.jnt_names.index(joint)]))

    def make():
        physics = BatchedPhysics.from_spec(spec, n, buffer_size=20, library=emu_library)
        physics.set_cpg(net)
        physics.set_cpg_state(net['phase0'], net['amplitude0'])
        return physics
    envs = [0, 3]
    A, C = make(), make()
    A.reset(qpos0, qvel0)
    A.step(7)
    spring_before = A.qpos_spring
    A.reset_envs(envs, qpos0[envs], qvel0[envs])
    phase, amp = A.cpg_state()
    assert np.array_equal(phase[envs], np.asarray(net['phase0'], np.float32)[envs].astype(np.float64))
    assert np.array_equal(amp[envs], np.broadcast_to(np.asarray(net['amplitude0'], np.float32), amp.shape)[envs])
    assert not np.array_equal(phase[1], np.asarray(net['phase0'], np.float32)[1])
    # qpos_spring is kept (the next step's sequence rows set the driven ones)
    assert np.array_equal(A.qpos_spring, spring_before)
    C.reset(qpos0, qvel0)
    for physics in (A, C):
        physics.step(9)
    identical, worst = differences(
        [(A.qpos[envs], C.qpos[envs]), (A.qvel[envs], C.qvel[envs]), (A.qpos_spring[envs], C.qpos_spring[envs])]
        + [(A.cpg_state()[i][envs], C.cpg_state()[i][envs]) for i in (0, 1)]
        + [(getattr(A.export_farms(e).sensors, k).array, getattr(C.export_farms(e).sensors, k).array)
           for e in envs for k in KINDS])
    assert identical, worst
    assert np.abs(A.qpos_spring[envs][:, [7 + 5, 7 + 6]] - model.qpos_spring[[7 + 5, 7 + 6]]).max() > 1e-3


def test_ground_to_water_clears_constraint_columns(emu_library):
    """An environment in ground contact restarted high above the ground: while the ring wraps, the
    contacts rows and the joint limit force of its rows are exactly zero (as test_ring_wrap)."""
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.layout import sc
    n, ring = 4, 5
    spec, model, qpos0, qvel0, ctrl = make_case('salamander', n, qvel_scale=0.05, ctrl_scale=0.1)
    physics = BatchedPhysics.from_spec(spec, n, buffer_size=ring, library=emu_library)
    physics.reset(qpos0, qvel0)
    physics.set_ctrl(ctrl)
    physics.step(8)
    logs = physics.log_arrays()
    assert np.abs(logs['contacts'][2]).max() > 0              # in contact before the restart
    high = qpos0[2].copy()
    high[2] += 50.0                                           # far above the ground: falls, no contact
    physics.reset_envs([2], high[None], np.zeros((1, model.nv)))
    for chunk in (3, 4, 6):
        physics.step(chunk)
        ours = physics.log_arrays(env=2)                      # the episode's rows
        assert not ours['contacts'].any() and not ours['joints'][..., sc.joint_limit_force].any()
        assert not physics.export_farms(2).sensors.contacts.array.any()
        if physics.iteration - 8 >= ring - 1:                 # every ring row is the episode's
            logs = physics.log_arrays()
            assert not logs['contacts'][2].any() and not logs['joints'][2][..., sc.joint_limit_force].any()
    assert physics.last_pending == n - 1                      # the others are still on the ground


def test_sub_steps(emu_library):
    """log_stride > 1: a restart at a full step; the export (full-step rows) matches a fresh batch."""
    sc = Scenario(emu_library, 'salamander_swim', 5, envs=[1, 2], k1=3, k2=4, ring=6, log_stride=3)
    for e in sc.envs:
        assert sc.A.episode_start()[e] == 9
        xa, xc = sc.A.export_farms(e), sc.C.export_farms(e)
        la, lc = sc.A.log_arrays(env=e), sc.C.log_arrays(env=e)
        for k in KINDS:
            assert np.array_equal(getattr(xa.sensors, k).array, getattr(xc.sensors, k).array), k
            assert np.array_equal(la[k], lc[k]), k
    assert np.array_equal(sc.A.qpos[sc.envs], sc.C.qpos[sc.envs])


# ------------------------------------------------------------------------------------ GPU
def gpu_paths():
    """(label, env vars, setup, n_envs): every path the launch can pick."""
    return [
        ('regular', {'FARMS_B200_FAST_BLOCK': '32', 'FARMS_B200_FAST_SLIM': '0', 'FARMS_B200_FAST_SPLIT': '0'},
         None, 'salamander_swim', 200),
        ('slim', {'FARMS_B200_FAST_BLOCK': '32', 'FARMS_B200_FAST_WPB': '1'}, lambda p: p.set_fast_slim(1),
         'salamander_swim', 200),
        ('slim_multi', {'FARMS_B200_FAST_BLOCK': '32', 'FARMS_B200_FAST_WPB': '7'}, lambda p: p.set_fast_slim(7),
         'salamander_swim', 500),
        ('split', {'FARMS_B200_FAST_BLOCK': '32'}, lambda p: p.set_fast_split(True), 'salamander_swim', 64),
        ('lean_off', {'FARMS_B200_FAST_BLOCK': '32', 'FARMS_B200_FAST_LEAN': '0'}, None, 'swimmer8', 100),
        ('lean_on', {'FARMS_B200_FAST_BLOCK': '32'}, None, 'swimmer8', 100),
        ('con16', {'FARMS_B200_FAST_BLOCK': '16', 'FARMS_B200_CON_SPLIT': '0'}, None, 'salamander', 64),
        ('con32', {'FARMS_B200_FAST_BLOCK': '32', 'FARMS_B200_CON_SPLIT': '0'}, None, 'salamander', 64),
        ('con_split16', {'FARMS_B200_FAST_BLOCK': '16', 'FARMS_B200_CON_SPLIT': '1'}, None, 'salamander', 64),
        ('con_split32', {'FARMS_B200_FAST_BLOCK': '32', 'FARMS_B200_CON_SPLIT': '1'}, None, 'salamander', 64),
        ('team', {}, lambda p: p.set_fast_path(False), 'salamander_swim', 64),
        ('team_con', {}, lambda p: p.set_constraint_path(False), 'salamander', 64),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize('label,env,setup,name,n_envs', gpu_paths(), ids=[p[0] for p in gpu_paths()])
def test_gpu_parity(cuda_library, monkeypatch, label, env, setup, name, n_envs):
    """Restarted environments against a fresh batch and the others against a never-restarted one,
    on each kernel path.  The restarted batch runs the ENVP = 1 kernels (the episode clock is bound), the
    two reference batches the entry points: a separate compilation of the same arithmetic, held to
    1e-6 relative (the SLIM MULTI layout differs by a few ulp, DESIGN section 4); the team kernel
    is one compilation: the same bits."""
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    rng = np.random.default_rng(1)
    envs = sorted(set(int(e) for e in rng.choice(n_envs, size=max(3, n_envs//10), replace=False)) | {0, n_envs - 1})
    sc = Scenario(cuda_library, name, n_envs, envs=envs, k1=8, k2=16, ring=11, setup=setup, chunks=[5, 11])
    if label.startswith('con') or label == 'team_con':
        assert sc.A.last_pending > 0
    compare(sc, exact=label == 'team', tol=1e-5 if label == 'slim_multi' else 1e-6)


def check_hand_over_mid_launch(library, n, tol):
    """Restarted swimming environments start just inside a joint limit that their position actuator
    pulls them through after a few steps (fastpath_cases.hand_over_case): the unconstrained ENVP = 1 kernel
    hands them over to the constrained one in the middle of the launch.  The wave controller (on
    the leg joints, so that it does not hold the driven body joints) keeps the episode clock bound."""
    import fastpath_cases
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.models import travelling_wave_parameters
    spec, model, q_hand, v_hand, ctrl = fastpath_cases.hand_over_case('salamander_swim', n)
    _, _, qpos0, qvel0, _ = make_case('salamander_swim', n)
    joints, _, freq, lag = travelling_wave_parameters(spec)
    legs = [i for i, j in enumerate(joints) if 'leg' in j]

    def make():
        physics = BatchedPhysics.from_spec(spec, n, buffer_size=17, library=library)
        physics.set_env_phase(np.linspace(0, 6, n))
        physics.set_wave_controller([model.actuator_id(f'actuator_position_{joints[i]}') for i in legs],
                                    np.full(len(legs), 0.2), freq[legs], lag[legs])
        return physics
    envs = list(range(0, n, 3))
    A, C = make(), make()
    A.reset(qpos0, qvel0)
    A.step(9)
    A.reset_envs(envs, q_hand[envs], v_hand[envs])
    start_q, start_v = qpos0.copy(), qvel0.copy()
    start_q[envs], start_v[envs] = q_hand[envs], v_hand[envs]
    C.reset(start_q, start_v)
    for physics in (A, C):
        physics.set_ctrl(ctrl)
        physics.step(16)
    assert 0 < A.last_pending < n, A.last_pending
    identical, worst = differences([(A.qpos[envs], C.qpos[envs]), (A.qvel[envs], C.qvel[envs])] +
                                   [(getattr(A.export_farms(e).sensors, k).array, getattr(C.export_farms(e).sensors, k).array)
                                    for e in envs[:6] for k in KINDS])
    print('hand-over', A.last_pending, 'bit-identical' if identical else f'{worst:.1e}')
    if tol == 0:
        assert identical, worst
    assert worst <= tol, worst


def test_hand_over_mid_launch(emu_library):
    check_hand_over_mid_launch(emu_library, 12, 0)


@pytest.mark.gpu
def test_gpu_hand_over_mid_launch(cuda_library):
    check_hand_over_mid_launch(cuda_library, 70, 1e-6)


@pytest.mark.gpu
def test_gpu_device_mask_matches_host_list(cuda_library):
    """fb_reset_envs_where with a mask computed in torch on the engine's stream (from flags and
    the state) gives what the host list gives."""
    import ctypes as ct
    import torch
    n = 256
    spec, model, qpos0, qvel0, _ = make_case('salamander_swim', n)
    phase = np.random.default_rng(2).uniform(0, 2*np.pi, n)
    rows_q = np.tile(model.key_qpos, (n, 1))
    rows_q[:, 7:] += 0.05
    rows_v = np.zeros((n, model.nv))
    out = []
    for device in (True, False):
        physics = wave_physics(cuda_library, spec, model, n, 9, phase)
        physics.reset(qpos0, qvel0)
        physics.step(8)
        if device:
            ptr = ct.c_void_p()
            physics.lib.fb_device_ptr_stream(physics._handle, ct.byref(ptr))
            stream = torch.cuda.ExternalStream(ptr.value)
            with torch.cuda.stream(stream):
                flags = torch.as_tensor(physics.device_array(physics.state_view.flags_dev, (n,), '<i4'), device='cuda')
                qpos = torch.as_tensor(physics.device_array(physics.state_view.qpos_dev, (n, model.nq)), device='cuda')
                mask = ((flags & 1) != 0) | (qpos[:, 0] > float(np.median(physics.qpos[:, 0])))
                q = torch.as_tensor(rows_q, dtype=torch.float32, device='cuda')
                v = torch.as_tensor(rows_v, dtype=torch.float32, device='cuda')
                physics.reset_envs(mask, q, v)
                physics.step(8, sync=False)
            envs = np.flatnonzero(mask.cpu().numpy())
        else:
            physics.reset_envs(envs, rows_q[envs], rows_v[envs])
            physics.step(8)
        physics.synchronize()
        out.append((physics.qpos, physics.qvel, physics.episode_start(), physics.log_arrays(),
                    [physics.export_farms(e) for e in envs[:4]]))
    assert 0 < len(envs) < n
    (qa, va, sa, la, xa), (qb, vb, sb, lb, xb) = out
    assert np.array_equal(qa, qb) and np.array_equal(va, vb) and np.array_equal(sa, sb)
    assert np.array_equal(sa[envs], [8]*len(envs))
    for k in KINDS:
        assert np.array_equal(la[k], lb[k]), k
        for a, b in zip(xa, xb):
            assert np.array_equal(getattr(a.sensors, k).array, getattr(b.sensors, k).array), k


@pytest.mark.gpu
def test_gpu_pipelined_host_calls(cuda_library):
    """fb_step_host_async with a restart between two calls: the rows the first call gathered are
    those of a batch without the restart, and the second call's ctrl drives the restarted
    environments."""
    from farms_mujoco_b200.engine import BatchedPhysics
    from farms_mujoco_b200.layout import sc
    n, steps = 128, 8
    spec, model, qpos0, qvel0, ctrl = make_case('salamander_swim', n)
    nl, nj = len(spec.links_names), len(spec.joints_names)
    envs = [3, 40, 41, 127]
    ctrl32 = np.ascontiguousarray(ctrl, dtype=np.float32)
    ctrl2 = np.ascontiguousarray(ctrl32[::-1])
    results = []
    for restart in (True, False):
        physics = BatchedPhysics.from_spec(spec, n, buffer_size=4, library=cuda_library)
        physics.reset(qpos0, qvel0)
        links = [np.zeros((n, nl, 20), np.float32) for _ in range(2)]
        joints = [np.zeros((n, nj, sc.joint_size), np.float32) for _ in range(2)]
        physics.step_host(steps, ctrl=ctrl32, links_row=links[0], joints_row=joints[0], pipelined=True)
        if restart:
            physics.reset_envs(envs, qpos0[envs], qvel0[envs])
        physics.step_host(steps, ctrl=ctrl2, links_row=links[1], joints_row=joints[1], pipelined=True)
        physics.host_wait()
        results.append((links, joints, physics.qpos))
    (la, ja, qa), (lb, jb, qb) = results
    assert np.array_equal(la[0], lb[0]) and np.array_equal(ja[0], jb[0])
    fresh = BatchedPhysics.from_spec(spec, n, buffer_size=4, library=cuda_library)
    fresh.reset(qpos0, qvel0)
    fresh.step_host(steps, ctrl=ctrl2)
    others = [e for e in range(n) if e not in envs]
    assert np.array_equal(qa[others], qb[others])
    identical, worst = differences([(qa[envs], fresh.qpos[envs]), (la[1][envs], fresh.log_arrays()['links'][envs, steps % 4])])
    assert identical, worst


@pytest.mark.gpu
def test_gpu_scale(cuda_library):
    """65,536 swimming SALAMANDERs (the headline configuration), 10 % restarted through the device
    mask before each of 20 launches of 16 steps: no non-finite state, and sampled restarted
    environments equal the same environments of a fresh batch."""
    import torch
    from farms_mujoco_b200 import models, mjcf_subset
    from farms_mujoco_b200.sharding import synthetic_inputs
    n, steps, launches = 65536, 16, 20
    spec = models.MODELS['salamander_swim']()
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    qpos0, qvel0, phase = synthetic_inputs(model, np.arange(n))
    physics = wave_physics(cuda_library, spec, model, n, steps + 1, phase)
    physics.reset(qpos0, qvel0)
    assert physics.fast_slim == 7
    q0 = torch.as_tensor(qpos0, dtype=torch.float32, device='cuda')
    v0 = torch.as_tensor(qvel0, dtype=torch.float32, device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(5)
    last = None
    for _ in range(launches):
        mask = torch.rand(n, device='cuda', generator=gen) < 0.1
        torch.cuda.synchronize()
        physics.reset_envs(mask, q0, v0)
        physics.step(steps)
        last = mask.cpu().numpy()
    assert not (physics.flags & 1).any()
    assert physics.iteration == steps*launches
    start = physics.episode_start()
    restarted = np.flatnonzero(last)
    assert np.array_equal(start[restarted], [steps*(launches - 1)]*len(restarted))
    sample = restarted[np.linspace(0, len(restarted) - 1, 8).astype(int)]
    fresh = wave_physics(cuda_library, spec, model, n, steps + 1, phase)
    fresh.reset(qpos0, qvel0)
    fresh.step(steps)
    identical, worst = differences([(physics.qpos[sample], fresh.qpos[sample]), (physics.qvel[sample], fresh.qvel[sample])] +
                                   [(getattr(physics.export_farms(int(e)).sensors, k).array,
                                     getattr(fresh.export_farms(int(e)).sensors, k).array) for e in sample[:3] for k in KINDS])
    print('65536 envs:', 'bit-identical' if identical else f'{worst:.1e}')
    assert worst < 1e-5, worst
