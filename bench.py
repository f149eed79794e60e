#!/usr/bin/env python
"""Benchmark of the hot path: env-steps/s of the fused FARMS step on B200.

Contract (one JSON line on stdout, rank 0):
  python bench.py --gpus N --steps K --warmup W            our arm (CUDA)
  python bench.py --impl reference --gpus N --steps K ...   CPU arm (oracle port)
  python bench.py ... --dump-outputs DIR                    also writes the last timed launch's
                                                            outputs to DIR/*.npy (dump_outputs)

Workload (config.workload): swimming salamander (28 links, nv=33) with
hydrodynamic drag + buoyancy and full sensor logging (links/joints/contacts/
xfrc), the 65,536-environment sweep BASELINE.json's metric is quoted on
(configs[4]): 65,536 environments per GPU, N GPUs step N x 65,536 independent
environments (weak scaling, no data-path collective).  ``--total-envs 65536`` is the
same sweep with the environments sharded over the GPUs (strong scaling);
``--envs-per-gpu 16384`` is configs[2].  One bench "step" = one launch of the fused
kernels advancing every environment by ``--inner`` physics steps.

value    : device-timed (CUDA events on the engine's stream, max over ranks),
           state resident in HBM.
e2e      : the same through BatchedPhysics.step_host on pinned HOST buffers, every launch:
           ctrl of the controlled actuators uploaded (evaluated by a host-side controller),
           the last joints row (4 written columns) and the head link's pose downloaded;
           e2e.full_log_export = rate of the streamed export of the FULL log (fb_export_rows).
roofline : algorithmic log bytes / launch time against measured HBM, plus the FP32 side
           (``fp32``); ``bound`` is the larger of the two fractions.
cpu_baseline / --impl reference: the oracle port on every host core (oracle/farms_loop.c: fp64 C
           restatement of mj_step + the farms glue), a bounded sample of the same workload.
extra    : (N = 1) device-timed lines of BASELINE.json's other configurations.
"""

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

_JSON_OUT = sys.stdout

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'env-steps/sec (box, device-timed) at 1/2/4/8 B200 vs ref CPU on host cores'
WORKLOAD = 'salamander_swim'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--envs-per-gpu', type=int, default=65536,
                    help='BASELINE.json config 5 at N = 1: 65,536 swimming salamanders on one B200 (config 3 is '
                         '--envs-per-gpu 16384)')
    ap.add_argument('--total-envs', type=int, default=0,
                    help='strong-scaling mode: this many environments in total, sharded evenly over the '
                         'GPUs (BASELINE.json north_star: 65,536 in total, 8,192 per GPU at N = 8); 0 = weak '
                         'scaling with --envs-per-gpu on every GPU')
    ap.add_argument('--e2e-links', default='head', choices=['head', 'pose', 'full'],
                    help="e2e arm, links rows downloaded per launch: 'head' = CoM position + orientation of the "
                         "first link (what a controller steering by the head pose reads), 'pose' = the same 7 "
                         "columns of every link, 'full' = all 20 columns of every link")
    ap.add_argument('--no-export', action='store_true', help='skip the full-log export measurement')
    ap.add_argument('--no-other-configs', action='store_true',
                    help="skip the short device-timed runs of BASELINE.json's other configurations "
                         "(reported under 'extra' at N = 1)")
    ap.add_argument('--inner', type=int, default=16, help='physics steps per launch')
    ap.add_argument('--ring', type=int, default=64, help='log ring rows per env')
    ap.add_argument('--model', default=WORKLOAD)
    ap.add_argument('--team', type=int, default=0)
    ap.add_argument('--cpu-seconds', type=float, default=12.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-fast', action='store_true', help='team kernel only (comparison runs)')
    ap.add_argument('--team-constraints', action='store_true',
                    help='hand-overs (limits / contacts) go to the team kernel instead of the per-thread '
                         'constrained kernel (comparison runs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed launch computed as DIR/<name>.npy '
                         '(float32): qpos, qvel and the log rows the launch wrote (links, joints, contacts, '
                         'xfrc) of a fixed seeded sample of the environments (rank 0), at most 60 MiB in all')
    return ap.parse_args()


# ------------------------------------------------------------------ inputs
from farms_mujoco_b200.sharding import synthetic_inputs, gather_env_statistics, bind_host_to_device  # noqa: E402


def wave_controller(spec, model, amplitude=0.3):
    from farms_mujoco_b200.models import travelling_wave_parameters
    joints, amp, freq, lag = travelling_wave_parameters(spec, amplitude=amplitude)
    acts = [model.actuator_id(f'actuator_position_{j}') for j in joints]
    return acts, amp, freq, lag


# ------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, False, [], set()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:  # pylint: disable=broad-except
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
            getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:  # pylint: disable=broad-except
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for bit, name in names.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:  # pylint: disable=broad-except
                pass
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=2)
        return {
            'sm_mhz': float(np.median(self.samples)) if self.samples else None,
            'sm_max_mhz': self.max_mhz,
            'reasons': sorted(self.reasons),
        }


# ---------------------------------------------------------------- CPU arm
CPU_ENVS_PER_CORE = 64


def _cpu_worker(args):
    """One process = one host core advancing ``envs`` environments of the workload by ``inner``
    physics steps per bench step, on the oracle port: the fp64 C restatement of mj_step plus the
    farms glue in C (oracle/farms_loop.c: physics2data, cycontacts2data, drag_forces / the swimming
    callback, the travelling-wave controller), one C call per environment and bench step -- the
    reference's order per iteration (task.py:168-186, simulation.py:156), no interpreter inside.
    Returns the wall time of every bench step and the per-stage seconds."""
    model_name, envs, inner, steps, warmup, ring, first_env = args
    sys.path.insert(0, ROOT)
    from farms_mujoco_b200 import models, mjcf_subset
    from farms_mujoco_b200.data import AnimatData
    from farms_mujoco_b200.simulation.physics import FarmsTables
    from oracle.oracle import OraclePhysics
    from oracle import farms_oracle as fo
    spec = models.MODELS[model_name]()
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    data = AnimatData.from_sensors_names(model.timestep, 2, spec.links_names, spec.joints_names,
                                         spec.contacts_names, spec.xfrc_names)
    maps = fo.make_maps(model, data)
    tables = FarmsTables(model, data.sensors, maps['sensors'], spec.animat_options,
                         spec.arena_options, spec.simulation_options.units)
    qpos, qvel, phase = synthetic_inputs(model, np.arange(first_env, first_env + envs))
    joints, amp, freq, lag = wave_controller(spec, model)
    loops = []
    for e in range(envs):
        physics = OraclePhysics(model)
        physics.reset(keyframe_id=0)
        physics.data.qpos[:] = qpos[e]
        physics.data.qvel[:] = qvel[e]
        physics.forward()
        loops.append(fo.CompiledRollout(physics, spec, tables, ring, wave=(np.array(joints), amp, freq, lag),
                                        env_phase=phase[e]))
    times = []
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        for loop in loops:
            loop.run(inner, timed=k >= warmup)
        times.append(time.perf_counter() - t0)
    stage = np.sum([loop.stage_seconds for loop in loops], axis=0)
    return times[warmup:], stage.tolist()


def cpu_reference_run(model_name, inner, steps, warmup, ring=64, cores=None, envs_per_core=CPU_ENVS_PER_CORE):
    """The CPU arm: ``cores`` processes x ``envs_per_core`` environments, every bench step advances
    all of them by ``inner`` physics steps (the same per-environment work as one GPU bench step,
    on a bounded number of environments)."""
    import multiprocessing as mp
    cores = cores or os.cpu_count() or 1
    ctx = mp.get_context('spawn')
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(model_name, envs_per_core, inner, steps, warmup, ring, i*envs_per_core)
                                     for i in range(cores)])
    # the processes run side by side without a barrier between steps: the job is done when the
    # slowest core is, so a bench step costs the largest per-core total divided by the step count
    total_s = max(sum(t) for t, _ in res)
    env_steps = cores*envs_per_core*inner*steps
    stage = np.sum([st for _, st in res], axis=0)
    names = ('physics2data+contacts', 'swimming drag + xfrc', 'control', 'mj_step')
    return {
        'value': env_steps/total_s, 'unit': 'env-steps/s', 'cores': cores, 'kind': 'port',
        'per_core': env_steps/total_s/cores,
        'ms_per_step': 1e3*total_s/steps,
        'stage_share': {n: float(v/stage.sum()) for n, v in zip(names, stage)},
        'sample': (f'{cores} processes x {envs_per_core} envs of {model_name} x {steps} steps of {inner} physics '
                   f'steps ({env_steps} env-steps, {float(stage.sum()):.1f} s of CPU work): fp64 C restatement of '
                   'mj_step + the farms glue in C (oracle/farms_loop.c; CPU port, not MuJoCo)'),
    }


def cpu_baseline(model_name, seconds, inner=16, cores=None):
    """Bounded sample for the GPU line's ``cpu_baseline`` object: about ``seconds`` of wall time."""
    cores = cores or os.cpu_count() or 1
    probe = cpu_reference_run(model_name, inner, steps=2, warmup=1, cores=cores, envs_per_core=4)
    per_step = probe['ms_per_step']*1e-3*CPU_ENVS_PER_CORE/4
    steps = int(max(3, min(200, seconds/max(per_step, 1e-6))))
    return cpu_reference_run(model_name, inner, steps=steps, warmup=1, cores=cores)


def run_reference(args, rank, world):
    """``--impl reference``: the reference's CPU path for this metric, timed on the host cores.
    The reference itself (MuJoCo + dm_control + farms_core) cannot be installed here (DESIGN.md
    section 2), so this is the oracle port, all host threads, on a bounded sample of the same
    workload: every bench step advances cores x 64 environments by --inner physics steps."""
    if rank != 0:
        return
    base = cpu_reference_run(args.model, args.inner, args.steps, max(1, args.warmup), ring=args.ring)
    n_envs = base['cores']*CPU_ENVS_PER_CORE
    out = {
        'impl': 'reference', 'metric': METRIC, 'value': base['value'], 'unit': 'env-steps/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': base['ms_per_step'], 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': (f'{args.model}: bounded sample of {n_envs} envs ({base["cores"]} host cores x '
                                f'{CPU_ENVS_PER_CORE}), drag+buoyancy, full links/joints/contacts/xfrc log, '
                                'travelling-wave control'),
                   'n_envs': n_envs, 'physics_steps_per_step': args.inner},
        'cpu_baseline': base,
        'e2e': {'value': base['value'], 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(out), file=_JSON_OUT, flush=True)


# ---------------------------------------------------------------- roofline helpers
def csrc_sha():
    """Hash of the kernel sources: the committed ncu traffic figures are only quoted while the
    kernels they were captured on are the ones being benchmarked."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, 'farms_mujoco_b200', 'csrc')
    for name in sorted(os.listdir(csrc)):
        if name.endswith(('.h', '.cu')):
            with open(os.path.join(csrc, name), 'rb') as f:
                h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic(model_name, n_envs, inner):
    """DRAM bytes per launch of the dominant kernel from the committed ``ncu --set full`` capture
    (profiles/traffic.json), or None when there is none for this (workload, batch, steps) or when
    it was captured on other kernel sources than the ones in the tree."""
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if not os.path.exists(tpath):
        return None, 'no profiles/traffic.json'
    with open(tpath) as f:
        tj = json.load(f)
    rec = tj.get('by_workload', {}).get(f'{model_name}:{n_envs}:{inner}')
    if not rec:
        return None, 'no ncu capture for this (workload, batch, steps)'
    if rec.get('csrc_sha') != csrc_sha():
        return None, f'stale: captured on csrc {rec.get("csrc_sha")}, tree is {csrc_sha()}'
    return rec['dram_bytes_per_launch'], rec.get('source')


def written_bytes_per_env_step(spec, constrained):
    """Bytes the step kernels actually store per env-step (fp32): the columns that carry values.
    The farms joints row is 18 columns of which physics.py:481-524 writes 4 (two 8-byte pairs here,
    a third when a limit may be active); contacts rows only exist while a contact is possible.  The
    other columns are zeros the log holds from its allocation on."""
    nl, nj = len(spec.links_names), len(spec.joints_names)
    nc, nx = len(spec.contacts_names), len(spec.xfrc_names)
    return 80*nl + (24 if constrained else 16)*nj + (48*nc if constrained else 0) + 24*nx


def kernel_name(physics, handed_over, n_local):
    if not physics.fast_path:
        return f'fb_step_kernel<{physics.team_lanes}>'
    lean = int(physics.fast_lean)
    if 2*handed_over > n_local:
        if physics.constraint_path and physics.con_split and handed_over == n_local:
            return (f'fb_fastc_split_kernel<{physics.fast_path},{lean}> '
                    f'({len(physics.fast_split_schedule())} warps per {physics.fast_path} envs)')
        return (f'fb_fastc_kernel<{physics.fast_path},{lean}>' if physics.constraint_path
                else f'fb_step_kernel<{physics.team_lanes}>')
    if physics.fast_split:
        return f'fb_fast_split_kernel<{lean}> ({physics.fast_split} warps per 32 envs)'
    return f'fb_fast_kernel<{physics.fast_path},{int(physics.fast_slim > 0)},{int(physics.fast_slim > 1)},{lean}>'


def roofline_objects(args_model, spec, physics, n_local, inner, k_ms, per_gpu_rate, handed_over, peaks, device):
    """The ``roofline`` and ``fp32`` objects of a bench line.  HBM side: algorithmic log bytes per
    launch / CUDA-event time of the launch against the measured copy bandwidth.  FP32 side
    (SURVEY 8d: "report both"): the oracle's instrumented op count of one mj_step
    (profiles/oracle_opcount.json) and the FADD / FMUL / FFMA the kernel executes (ncu) against the
    FFMA throughput the library measures on this device.  ``bound`` names the roof the kernel
    sits closer to."""
    b_log = physics.log_bytes_per_env_step
    peak = float(peaks.get('hbm_gbs', 6650.0))
    achieved = n_local*inner*b_log/(k_ms*1e-3)/1e9
    constrained = 2*handed_over > n_local
    b_written = written_bytes_per_env_step(spec, constrained)
    traffic, traffic_source = measured_traffic(args_model, n_local, inner)
    fp32 = None
    try:
        from farms_mujoco_b200.engine import measure_fp32_peak
        fp32_peak = measure_fp32_peak(device)
        with open(os.path.join(ROOT, 'profiles', 'oracle_opcount.json')) as f:
            oc = json.load(f)
        rec = oc['models'].get(args_model)
        if rec:
            fp32 = {
                'peak_tflops': fp32_peak, 'peak_source': 'fb_measure_fp32_peak (FFMA micro-benchmark, this run)',
                'oracle_flop_per_env_step': rec['flop'],
                'oracle_equivalent_tflops': per_gpu_rate*rec['flop']*1e-12,
                'oracle_equivalent_frac': per_gpu_rate*rec['flop']*1e-12/fp32_peak,
                'executed_flop_per_env_step': oc.get('executed_flop_per_env_step', {}).get(args_model),
            }
            if fp32['executed_flop_per_env_step'] and not constrained:
                fp32['executed_tflops'] = per_gpu_rate*fp32['executed_flop_per_env_step']*1e-12
                fp32['executed_frac'] = fp32['executed_tflops']/fp32_peak
    except (OSError, KeyError, ValueError) as exc:
        fp32 = {'error': str(exc)}
    hbm_frac = achieved/peak
    fp32_frac = (fp32 or {}).get('oracle_equivalent_frac') or 0.0
    roofline = {
        'bound': 'hbm' if hbm_frac >= fp32_frac else 'fp32',
        'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': hbm_frac,
        'traffic': traffic, 'traffic_source': traffic_source,
        'kernel': kernel_name(physics, handed_over, n_local),
        'kernel_ms': k_ms,
        'algorithmic_bytes_per_env_step': b_log,
        'written_bytes_per_env_step': b_written,
        'frac_written_bytes': n_local*inner*b_written/(k_ms*1e-3)/1e9/peak,
        'fp32_frac_oracle_equivalent': fp32_frac,
        'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured)' if peaks else 'fallback 6650',
        'note': ('achieved = algorithmic log bytes (B_log, SURVEY 8d: every column of every row) per launch / '
                 'mean CUDA-event time of a launch on the engine stream; written_bytes counts only the columns '
                 'that carry values (the constant-zero columns are not stored again); the kernels are '
                 'issue/latency bound, below both roofs: see profiles/ for issue-slot utilisation'),
    }
    return roofline, fp32


def short_device_run(name, n_envs, inner, ring, steps, warmup, device, peaks, amplitude=0.3):
    """Device-timed run of another BASELINE.json configuration on this GPU (no e2e, no CPU arm).
    ``amplitude`` > 1 drives the body joints into their +-1 rad limits: the mixed regime in which the
    unconstrained kernel hands environments over to the constrained one in the middle of a launch."""
    import ctypes
    import torch
    from farms_mujoco_b200 import models, mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    spec = models.MODELS[name]()
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    qpos0, qvel0, phase = synthetic_inputs(model, np.arange(n_envs))
    physics = BatchedPhysics.from_spec(spec, n_envs, buffer_size=ring, device=device)
    physics.set_env_phase(phase)
    physics.set_wave_controller(*wave_controller(spec, model, amplitude))
    physics.reset(qpos0, qvel0)
    stream_ptr = ctypes.c_void_p()
    physics._check(physics.lib.fb_device_ptr_stream(physics._handle, ctypes.byref(stream_ptr)))
    stream = torch.cuda.ExternalStream(stream_ptr.value, device=device)
    for _ in range(warmup):
        physics.step(inner, sync=False)
    physics.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = physics.launch_count()
    with torch.cuda.stream(stream):
        ev0.record()
        for _ in range(steps):
            physics.step(inner, sync=False)
        ev1.record()
    physics.synchronize()
    ms = ev0.elapsed_time(ev1)
    launches = physics.launch_count() - launches0
    k_ms = []
    for _ in range(3):
        physics.step(inner, sync=True)
        k_ms.append(physics.last_step_ms())
    handed_over = physics.last_pending if physics.fast_path else n_envs
    value = n_envs*inner*steps/(ms*1e-3)
    roofline, fp32 = roofline_objects(name, spec, physics, n_envs, inner, float(np.mean(k_ms)), value,
                                      handed_over, peaks, device)
    flags = physics.flags
    out = {
        'workload': (f'{name}: {n_envs} envs on 1 GPU, full log, on-device travelling-wave control'
                     + ('' if amplitude == 0.3 else f', wave amplitude {amplitude} rad (joint limits at +-1: mixed regime)')),
        'value': value, 'unit': 'env-steps/s', 'ms_per_step': ms/steps, 'steps': steps, 'warmup': warmup,
        'physics_steps_per_step': inner, 'gpu_launches': int(launches),
        'handed_over_envs_last_launch': int(handed_over), 'diverged_envs': int(np.count_nonzero(flags & 1)),
        'roofline': roofline, 'fp32': fp32,
    }
    physics.close()
    return out


DUMP_BYTES = 60 << 20


def dump_outputs(physics, inner, out_dir):
    """``--dump-outputs``: the state ``qpos`` [S, nq], ``qvel`` [S, nv] and the log rows the last
    launch wrote, ``<kind>`` [S, rows, n_items, n_cols], float32 as the engine holds them, so that
    two builds can be compared output for output on the same inputs.  The S environments are
    ``np.random.default_rng(0).choice(n_envs, S, replace=False)`` in ascending order, S as large
    as DUMP_BYTES allows."""
    rows = min(inner, physics.buffer_size)
    first = physics.iteration - rows + 1          # step j writes ring row (j + 1) % ring
    per_env = 4*(physics.model.nq + physics.model.nv) + rows*physics.log_bytes_per_env_step
    n_sample = min(physics.n_envs, DUMP_BYTES//per_env)
    envs = np.sort(np.random.default_rng(0).choice(physics.n_envs, n_sample, replace=False))
    out = {'qpos': physics.qpos[envs], 'qvel': physics.qvel[envs]}
    for kind in ('links', 'joints', 'contacts', 'xfrc'):
        out[kind] = np.stack([physics.log_row(kind, (first + r) % physics.buffer_size)[envs]
                              for r in range(rows)], axis=1)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), arr)


# ---------------------------------------------------------------- GPU arm
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from farms_mujoco_b200 import models, mjcf_subset
    from farms_mujoco_b200.engine import BatchedPhysics
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the engine has no CPU fallback)')
    torch.cuda.set_device(local_rank)
    # host side of the e2e arm on the GPU's own NUMA node (pinned buffers, controller threads)
    bound = None if os.environ.get('FARMS_B200_NO_BIND') else bind_host_to_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    spec = models.MODELS[args.model]()
    model = mjcf_subset.parse_mjcf(spec.mjcf)
    if args.total_envs:
        if args.total_envs % world:
            raise SystemExit('--total-envs must be a multiple of the number of GPUs')
        n_local = args.total_envs//world
    else:
        n_local = args.envs_per_gpu
    env_ids = np.arange(rank*n_local, (rank + 1)*n_local)
    qpos0, qvel0, phase = synthetic_inputs(model, env_ids)
    physics = BatchedPhysics.from_spec(spec, n_local, buffer_size=args.ring, device=local_rank,
                                       team_lanes=args.team)
    physics.set_env_phase(phase)
    physics.set_wave_controller(*wave_controller(spec, model))
    if args.no_fast:
        physics.set_fast_path(False)
    if args.team_constraints:
        physics.set_constraint_path(False)
    physics.reset(qpos0, qvel0)

    stream_ptr = __import__('ctypes').c_void_p()
    physics._check(physics.lib.fb_device_ptr_stream(physics._handle, __import__('ctypes').byref(stream_ptr)))
    stream = torch.cuda.ExternalStream(stream_ptr.value, device=local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(stream):
            ev0.record()
            for _ in range(steps):
                fn()
            ev1.record()
        physics.synchronize()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device='cuda')
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident arm
    for _ in range(args.warmup):
        physics.step(args.inner, sync=False)
    physics.synchronize()
    launches0 = physics.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    kernel_ms = []

    def one():
        physics.step(args.inner, sync=False)

    total_ms = timed(one, args.steps)
    clocks = sampler.summary()
    launches = physics.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(physics, args.inner, args.dump_outputs)
    # per-launch kernel time from the engine's own CUDA events (recorded on the engine's stream
    # around the launch pair): mean over a few more launches, each read back before the next
    for _ in range(5):
        physics.step(args.inner, sync=True)
        kernel_ms.append(physics.last_step_ms())
    env_steps = n_local*world*args.inner*args.steps
    value = env_steps/(total_ms*1e-3)
    handed_over = physics.last_pending if physics.fast_path else n_local

    # ---- end-to-end arm on pinned host buffers
    e2e = None
    if not args.no_e2e:
        nl, njf = len(spec.links_names), len(spec.joints_names)
        # three sets of pinned host buffers: the engine's pipelined step_host overlaps the
        # download of launch i with the kernels of launch i+1 (include/farms_b200.h); the third
        # set lets the host enqueue launch i+1 (and its ctrl upload) while launch i still runs
        NSETS = 3
        # the links row comes down as CoM position + orientation (7 of the 20 columns: what a host
        # controller steering by pose reads; the velocities stay in the device log) unless
        # --e2e-full-links asks for the whole row
        lcols = list(range(20)) if args.e2e_links == 'full' else list(range(7))
        litems = [0] if args.e2e_links == 'head' else list(range(nl))
        physics.set_host_link_columns(None if args.e2e_links == 'full' else lcols)
        physics.set_host_link_items(litems if args.e2e_links == 'head' else None)
        links_host = [torch.empty((n_local, len(litems), len(lcols)), dtype=torch.float32).pin_memory() for _ in range(NSETS)]
        # the joints row comes down as the four columns the path writes (position, velocity,
        # torque, limit force); physics.py:481-524 leaves the other 14 of the 18 zero
        from farms_mujoco_b200.layout import sc
        jcols = [sc.joint_position, sc.joint_velocity, sc.joint_torque, sc.joint_limit_force]
        physics.set_host_joint_columns(jcols)
        joints_host = [torch.empty((n_local, njf, len(jcols)), dtype=torch.float32).pin_memory() for _ in range(NSETS)]
        physics.set_wave_controller(None, None, None, None)   # ctrl now comes from the host
        acts, amp, freq, lag = wave_controller(spec, model)
        acts_t = torch.as_tensor(np.array(acts))
        amp_t, freq_t = torch.as_tensor(amp, dtype=torch.float32), torch.as_tensor(freq, dtype=torch.float32)
        lag_t = torch.as_tensor(lag, dtype=torch.float32)
        phase_t = torch.as_tensor(phase, dtype=torch.float32)[:, None]
        # amp sin(a - lag + phase) = [amp sin(a - lag)] cos(phase) + [amp cos(a - lag)] sin(phase):
        # the per-environment factors are constant, so a call costs two multiply-adds per entry
        cos_ph, sin_ph = torch.cos(phase_t), torch.sin(phase_t)
        # ctrl goes up as the controlled actuators only (the position actuators the controller
        # writes, task.py:309-321): [n_envs, n_controlled] instead of [n_envs, nu]; the velocity
        # and motor actuators keep their (zero) ctrl on the device
        compact = len(acts) <= 32
        if compact:
            physics.set_host_ctrl_columns(acts)
        ctrl_host = [torch.zeros((n_local, len(acts) if compact else model.nu), dtype=torch.float32).pin_memory()
                     for _ in range(NSETS)]
        wave_buf = torch.empty((n_local, len(acts)), dtype=torch.float32)
        if world > 1:
            # torchrun pins every rank to one OpenMP thread; the host-side controller may use its share
            torch.set_num_threads(max(1, min(len(bound) if bound else 1 << 30, (os.cpu_count() or world)//world)))
        checksum = [0.0]
        calls = [0]
        pending = [None]*NSETS

        def one_host():
            # host-side controller of this outer iteration (task.py:288-321 analogue):
            # the same travelling wave, evaluated on the host and uploaded
            k = calls[0] % NSETS
            calls[0] += 1
            if pending[k] is not None:
                # the buffers of NSETS calls ago are complete once this call is allowed to reuse
                # them: consume the result (every step's rows are read on the host)
                physics.host_wait_call(pending[k])
                checksum[0] += float(links_host[k][0, 0, 0]) + float(joints_host[k][-1, 0, 0])
            t = physics.iteration*model.timestep
            arg = 2*np.pi*freq_t*t - lag_t
            out_buf = ctrl_host[k] if compact else wave_buf
            torch.mul(cos_ph, amp_t*torch.sin(arg), out=out_buf)
            out_buf.addcmul_(sin_ph, amp_t*torch.cos(arg))
            if not compact:
                ctrl_host[k].index_copy_(1, acts_t, wave_buf)
            pending[k] = physics.step_host(args.inner, ctrl=ctrl_host[k], links_row=links_host[k],
                                           joints_row=joints_host[k], pipelined=True)

        for _ in range(max(NSETS, args.warmup)):
            one_host()
        physics.host_wait()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            one_host()
        physics.host_wait()
        barrier()
        wall = torch.tensor([time.perf_counter() - t0], device='cuda')
        if world > 1:
            dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        links_host = links_host[(calls[0] - 1) % NSETS]
        ctrl_host, joints_host = ctrl_host[0], joints_host[0]
        e2e = {
            'value': env_steps/float(wall.item()), 'unit': 'env-steps/s',
            'h2d_bytes_per_step': int(ctrl_host.numel()*4*world),
            'd2h_bytes_per_step': int((links_host.numel() + joints_host.numel())*4*world),
            'checksum': float(links_host[:, 0, 0].double().sum()) + checksum[0],
            'pipelined': 'device->host copy of launch i overlaps the kernels of launch i+1 (fb_step_host_async, three host buffer sets); ctrl is fetched from pinned host memory by the SMs on an upload stream',
            'ctrl_up': (f'[n_envs, {len(acts)}] controlled (position) actuators of every launch, evaluated by a host-side '
                        'travelling-wave controller' if compact else '[n_envs, nu]'),
            'host_cpus_bound': len(bound) if bound else None,
            'rows_down': (f'of every launch, the last links row [n_envs, {len(litems)} link(s), {len(lcols)} columns'
                          + ('' if args.e2e_links == 'full' else ': CoM position + orientation')
                          + '] + the last joints row [n_envs, n_joints, 4 written columns: position, velocity, '
                          'torque, limit force]; the rest of the log stays on the device (full_log_export)'),
        }
        if world == 1 and not args.no_export:
            # streamed export of the FULL log (every column of every kind, the arrays the
            # reference saves, simulation.py:198-209): 4 ring rows of every environment
            rows = 4
            bufs = {k: torch.empty((rows, n_local, n_items, cols), dtype=torch.float32).pin_memory()
                    for k, n_items, cols in (('links', nl, 20), ('joints', njf, 18),
                                             ('contacts', len(spec.contacts_names), 12), ('xfrc', len(spec.xfrc_names), 6))}
            for k, buf in bufs.items():
                physics.export_rows(k, 0, 1, out=buf)            # warm-up (staging allocation)
            t0 = time.perf_counter()
            for k, buf in bufs.items():
                physics.export_rows(k, 0, rows, out=buf)
            dt = time.perf_counter() - t0
            nbytes = sum(b.numel()*4 for b in bufs.values())
            e2e['full_log_export'] = {
                'GB_per_s': nbytes/dt/1e9, 'bytes': nbytes, 'rows': rows,
                'env_steps_per_s_exportable': rows*n_local/dt,
                'note': 'fb_export_rows: ring rows -> dense pinned host arrays [rows, n_envs, n_items, n_cols], '
                        'gathers double-buffered against the device->host copies',
            }
            del bufs

    # ---- optional end-of-rollout gather of per-env statistics (NCCL)
    stats = torch.as_tensor(physics.qpos[:, :3].astype(np.float32), device='cuda')
    stats = gather_env_statistics(stats, world)
    all_flags = physics.flags
    flags = int(np.count_nonzero(all_flags & 1))
    solver_flags = int(np.count_nonzero(all_flags & 4))

    if rank == 0:
        b_log = physics.log_bytes_per_env_step
        peaks = {}
        try:
            with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
                peaks = json.load(f)
        except OSError:
            pass
        k_ms = float(np.mean(kernel_ms))
        roofline, fp32 = roofline_objects(args.model, spec, physics, n_local, args.inner, k_ms, value/world,
                                          handed_over, peaks, local_rank)
        out = {
            'metric': METRIC, 'value': value, 'unit': 'env-steps/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms/args.steps,
            'higher_is_better': True, 'scaling': 'strong' if args.total_envs else 'weak',
            'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic',
            'config': {
                'workload': (f'{args.model}: {n_local} envs/GPU x {world} GPU, drag+buoyancy, full '
                             'links/joints/contacts/xfrc log, on-device travelling-wave control'),
                'n_envs': n_local*world, 'physics_steps_per_step': args.inner, 'timestep': model.timestep,
                'nv': model.nv, 'nbody': model.nbody,
                'kernels': (('fb_fast_kernel (1 thread = 1 env, articulated-body recursion) then '
                             + ('fb_fastc_kernel (1 thread = 1 env, matrix-free Newton on the same recursion) '
                                'on the environments with an active limit / contact' if physics.constraint_path
                                else 'fb_step_kernel (lane team = 1 env, constraint solver) on the hand-overs'))
                            if physics.fast_path else 'fb_step_kernel only'),
                'fast_envs_per_block': physics.fast_path,
                'fast_slim_layout': bool(physics.fast_slim),
                'fast_lean_variant': bool(physics.fast_lean),
                'fast_split_warps': int(physics.fast_split),
                'constrained_split': bool(physics.con_split),
                'fast_warps_per_block': max(1, int(physics.fast_slim)),
                'fast_smem_bytes_per_env': physics.fast_smem_bytes_per_env,
                'handed_over_envs_last_launch': handed_over,
                'team_lanes': physics.team_lanes, 'team_smem_bytes_per_env': physics.smem_bytes_per_env,
                'l2_policy': (f'no flush: each step appends {n_local*args.inner*b_log/1e6:.0f} MB of new '
                              f'log rows to a {n_local*args.ring*b_log/1e9:.1f} GB ring (> 126 MB L2)'),
                'diverged_envs': flags, 'solver_pivot_clamped_envs': solver_flags,
            },
            'clocks': clocks,
            'e2e': e2e,
            'gpu_launches': int(launches),
            'fp32': fp32,
            'roofline': roofline,
        }
        if not args.no_cpu_baseline and world == 1:
            out['cpu_baseline'] = cpu_baseline(args.model, args.cpu_seconds, inner=args.inner)
        if world == 1 and not args.no_other_configs and args.model == WORKLOAD:
            # BASELINE.json's other configurations, device-timed on this GPU (parity cases with a
            # number attached; the headline stays the line's own value)
            physics.close()
            extra = []
            for name, n_envs, amplitude in (('salamander', 4096, 0.3), ('salamander_swim', 16384, 0.3),
                                            ('centipede', 8192, 0.3), ('salamander_swim', 8192, 0.3),
                                            ('salamander_swim', 16384, 1.3)):
                if name == args.model and n_envs == n_local and amplitude == 0.3:
                    continue
                try:
                    extra.append(short_device_run(name, n_envs, args.inner, 64, args.steps, args.warmup, local_rank,
                                                  peaks, amplitude))
                except Exception as exc:  # pylint: disable=broad-except
                    extra.append({'workload': f'{name}: {n_envs} envs', 'error': str(exc)})
            out['extra'] = {'other_configs': extra}
        print(json.dumps(out), file=_JSON_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner) write
    # to fd 1 too: everything but our line goes to stderr.
    global _JSON_OUT  # pylint: disable=global-statement
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    args = parse_args()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        if args.dump_outputs:
            raise SystemExit('--dump-outputs writes the outputs of the CUDA arm (--impl b200)')
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        raise SystemExit('launch N>1 with torch.distributed.run (one rank per GPU)')
    run_b200(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
