"""Batched physics over the C ABI (include/farms_b200.h).

``BatchedPhysics`` stands where dm_control's ``Physics`` stands in the reference
(farms_mujoco/simulation/simulation.py:53 ``mjcf.Physics.from_mjcf_model`` and
:156 ``env.step`` -> ``mj_step``): it owns the compiled model and the state of
``n_envs`` independent environments and advances all of them with one call.
There is no CPU fallback: construction raises when the CUDA library is missing
or no GPU is present.
"""

import ctypes as ct
import os

import numpy as np

from . import cabi
from .data import AnimatData
from .layout import sc
from .mjcf_subset import PAIR_MIN_FRICTION, candidate_friction, parse_mjcf
from .simulation.physics import FarmsTables, get_sensor_maps, get_physics2data_maps
from .units import SimulationUnitScaling

_PKG = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIBRARY = os.path.join(_PKG, 'libfarmsb200.so')

# name, restype, argtypes -- every symbol include/farms_b200.h declares
_H = ct.c_void_p
ABI_SYMBOLS = {
    'fb_last_error': (ct.c_char_p, []),
    'fb_abi_version': (ct.c_int, []),
    'fb_create': (ct.c_int, [ct.POINTER(cabi.FbModel), ct.POINTER(cabi.FbFarms), ct.c_int,
                             ct.c_int, ct.c_int, ct.c_int, ct.POINTER(_H)]),
    'fb_destroy': (None, [_H]),
    'fb_reset': (ct.c_int, [_H, cabi.c_double_p, cabi.c_double_p]),
    'fb_reset_envs': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32), cabi.c_double_p, cabi.c_double_p]),
    'fb_reset_envs_where': (ct.c_int, [_H, ct.c_void_p, ct.c_void_p, ct.c_void_p]),
    'fb_get_episode_start': (ct.c_int, [_H, cabi.c_int64_p]),
    'fb_set_ctrl': (ct.c_int, [_H, cabi.c_double_p]),
    'fb_set_qpos_spring': (ct.c_int, [_H, cabi.c_double_p]),
    'fb_set_ctrl_sequence': (ct.c_int, [_H, ct.c_void_p, ct.c_int]),
    'fb_set_env_phase': (ct.c_int, [_H, cabi.c_double_p]),
    'fb_set_wave_controller': (ct.c_int, [_H, ct.POINTER(cabi.FbWaveController)]),
    'fb_set_cpg': (ct.c_int, [_H, ct.POINTER(cabi.FbCpgNetwork)]),
    'fb_set_cpg_springrefs': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32), ct.POINTER(ct.c_int32), ct.POINTER(ct.c_int32),
                              cabi.c_double_p, cabi.c_double_p]),
    'fb_set_cpg_state': (ct.c_int, [_H, cabi.c_double_p, cabi.c_double_p]),
    'fb_get_cpg_state': (ct.c_int, [_H, cabi.c_double_p, cabi.c_double_p]),
    'fb_set_actuator_forcerange': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32), ct.POINTER(ct.c_int32), cabi.c_double_p]),
    'fb_set_water_velocity': (ct.c_int, [_H, ct.c_double, ct.c_double, ct.c_double]),
    'fb_set_swimming': (ct.c_int, [_H, ct.c_int, ct.c_int]),
    'fb_set_env_param': (ct.c_int, [_H, ct.c_int, cabi.c_double_p]),
    'fb_get_env_param': (ct.c_int, [_H, ct.c_int, cabi.c_double_p]),
    'fb_step': (ct.c_int, [_H, ct.c_int, ct.c_int, ct.c_int]),
    'fb_synchronize': (ct.c_int, [_H]),
    'fb_last_step_ms': (ct.c_int, [_H, ct.POINTER(ct.c_float)]),
    'fb_launch_count': (ct.c_int64, [_H]),
    'fb_log_view': (ct.c_int, [_H, ct.POINTER(cabi.FbLogView)]),
    'fb_state_view': (ct.c_int, [_H, ct.POINTER(cabi.FbStateView)]),
    'fb_derived_view': (ct.c_int, [_H, ct.POINTER(cabi.FbDerivedView)]),
    'fb_export_farms': (ct.c_int, [_H, ct.c_int, cabi.c_double_p, cabi.c_double_p,
                                   cabi.c_double_p, cabi.c_double_p]),
    'fb_host_wait': (ct.c_int, [_H]),
    'fb_set_host_joint_columns': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32)]),
    'fb_set_host_link_columns': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32)]),
    'fb_set_host_link_items': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32)]),
    'fb_set_host_ctrl_columns': (ct.c_int, [_H, ct.c_int, ct.POINTER(ct.c_int32)]),
    'fb_export_rows': (ct.c_int, [_H, ct.c_int, ct.c_int, ct.c_int, ct.c_void_p]),
    'fb_host_wait_slot': (ct.c_int, [_H, ct.c_int]),
    'fb_host_call_count': (ct.c_longlong, [_H]),
    'fb_host_wait_call': (ct.c_int, [_H, ct.c_longlong]),
    'fb_step_host': (ct.c_int, [_H, ct.c_void_p, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_void_p,
                                ct.c_void_p]),
    'fb_step_host_async': (ct.c_int, [_H, ct.c_void_p, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_void_p,
                                      ct.c_void_p]),
    'fb_copy_to_host': (ct.c_int, [_H, ct.c_void_p, ct.c_void_p, ct.c_int64]),
    'fb_copy_to_device': (ct.c_int, [_H, ct.c_void_p, ct.c_void_p, ct.c_int64]),
    'fb_set_fast_path': (ct.c_int, [_H, ct.c_int]),
    'fb_fast_path': (ct.c_int, [_H]),
    'fb_set_constraint_path': (ct.c_int, [_H, ct.c_int]),
    'fb_constraint_path': (ct.c_int, [_H]),
    'fb_fast_smem_bytes_per_env': (ct.c_int, [_H]),
    'fb_set_fast_slim': (ct.c_int, [_H, ct.c_int]),
    'fb_fast_slim': (ct.c_int, [_H]),
    'fb_set_fast_split': (ct.c_int, [_H, ct.c_int]),
    'fb_fast_split': (ct.c_int, [_H]),
    'fb_fast_split_blocks_per_sm': (ct.c_int, [_H]),
    'fb_set_con_split': (ct.c_int, [_H, ct.c_int]),
    'fb_con_split': (ct.c_int, [_H]),
    'fb_fast_split_schedule': (ct.c_int, [_H, ct.POINTER(ct.c_int32), ct.POINTER(ct.c_int32), ct.POINTER(ct.c_uint8)]),
    'fb_set_fast_lean': (ct.c_int, [_H, ct.c_int]),
    'fb_fast_lean': (ct.c_int, [_H]),
    'fb_last_pending': (ct.c_int, [_H, ct.POINTER(ct.c_int)]),
    'fb_measure_fp32_peak': (ct.c_int, [ct.c_int, ct.POINTER(ct.c_double)]),
    'fb_drag_forces': (ct.c_int, [ct.c_int, ct.c_int, cabi.c_double_p, cabi.c_double_p, cabi.c_double_p,
                                  cabi.c_double_p, cabi.c_double_p, ct.c_double, cabi.c_double_p,
                                  ct.c_double, ct.c_double, ct.c_int, cabi.c_double_p, ct.POINTER(ct.c_int32)]),
    'fb_team_lanes': (ct.c_int, [_H]),
    'fb_smem_bytes_per_env': (ct.c_int, [_H]),
    'fb_device_ptr_stream': (ct.c_int, [_H, ct.POINTER(ct.c_void_p)]),
}

_LIBS = {}


class EngineError(RuntimeError):
    """Raised for every non-zero return of the C ABI (message = fb_last_error)."""


def load_library(path=None):
    """dlopen the engine and bind every ABI symbol.  No fallback of any kind."""
    path = os.path.abspath(path or DEFAULT_LIBRARY)
    if path in _LIBS:
        return _LIBS[path]
    if not os.path.exists(path):
        raise EngineError(
            f'{path} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc, sm_100a).  The engine has no CPU fallback.')
    lib = ct.CDLL(path)
    for name, (restype, argtypes) in ABI_SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.fb_abi_version() != 2:
        raise EngineError('ABI version mismatch')
    _LIBS[path] = lib
    return lib


def measure_fp32_peak(device=0, library=None):
    """Measured FFMA throughput of ``device`` in TFLOP/s (``fb_measure_fp32_peak``)."""
    lib = load_library(library)
    out = ct.c_double()
    if lib.fb_measure_fp32_peak(int(device), ct.byref(out)) != 0:
        raise EngineError(lib.fb_last_error().decode())
    return float(out.value)


def drag_forces_rows(links, coefficients, mass, height, density, surface, water_velocity, viscosity,
                     gravity, use_buoyancy, xfrc, device=0, library=None):
    """``fb_drag_forces``: the reference's ``drag_forces`` (drag.pyx:152-268) on ``n`` link rows at
    once on the device, float64.  ``links`` [n, 20], ``coefficients`` [n, 2, 3] (or [n, 6]), ``mass``
    / ``height`` / ``density`` [n]; ``xfrc`` [n, 6] float64 C-contiguous is updated in place where the
    link is at or below the surface.  Returns the boolean ``applied`` [n] (drag_forces' return)."""
    lib = load_library(library)
    links = np.ascontiguousarray(links, dtype=np.float64)
    n = links.shape[0]
    if links.shape != (n, 20):
        raise ValueError('links must be [n, 20]')
    coef = np.ascontiguousarray(np.asarray(coefficients, dtype=np.float64).reshape(n, 6))
    per = [np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.float64), (n,))) for a in (mass, height, density)]
    wvel = np.ascontiguousarray(water_velocity, dtype=np.float64).reshape(3)
    if not (isinstance(xfrc, np.ndarray) and xfrc.dtype == np.float64 and xfrc.flags.c_contiguous
            and xfrc.shape == (n, 6)):
        raise ValueError('xfrc must be a C-contiguous float64 [n, 6] array (updated in place)')
    applied = np.zeros(n, dtype=np.int32)
    dp = lambda a: a.ctypes.data_as(cabi.c_double_p)
    if lib.fb_drag_forces(int(device), int(n), dp(links), dp(coef), dp(per[0]), dp(per[1]), dp(per[2]),
                          float(surface), dp(wvel), float(viscosity), float(gravity), int(bool(use_buoyancy)),
                          dp(xfrc), applied.ctypes.data_as(ct.POINTER(ct.c_int32))) != 0:
        raise EngineError(lib.fb_last_error().decode())
    return applied.astype(bool)


class _DeviceArray:
    """Zero-copy handle on an engine-owned device buffer (``__cuda_array_interface__``)."""

    def __init__(self, ptr, shape, typestr, owner):
        self.ptr, self.shape, self.typestr, self.owner = int(ptr), tuple(shape), typestr, owner
        self.__cuda_array_interface__ = {
            'shape': self.shape, 'typestr': typestr, 'data': (self.ptr, False), 'version': 2,
            'strides': None,
        }


def _ptr(p):
    return ct.cast(p, ct.c_void_p).value or 0


def _device_address(arr):
    """Device address of a CUDA array (``__cuda_array_interface__``, or a torch CUDA tensor's
    ``data_ptr()``); None for host data."""
    if hasattr(arr, 'data_ptr') and getattr(arr, 'is_cuda', False):
        return int(arr.data_ptr())
    cai = getattr(arr, '__cuda_array_interface__', None)
    return None if cai is None else int(cai['data'][0])


def _device_shape(arr):
    """(shape, typestr) of a CUDA array; it must be C-contiguous."""
    cai = arr.__cuda_array_interface__
    shape = tuple(int(d) for d in cai['shape'])
    strides = cai.get('strides')
    if strides is not None:
        item = int(cai['typestr'][2:])
        expect, acc = [], item
        for d in reversed(shape):
            expect.insert(0, acc)
            acc *= d
        if tuple(strides) != tuple(expect):
            raise ValueError('reset_envs: device arrays must be C-contiguous')
    return shape, cai['typestr']


class BatchedPhysics:
    """``n_envs`` copies of one compiled FARMS model stepping in lockstep."""
    # pylint: disable=too-many-instance-attributes,too-many-public-methods

    def __init__(self, model, n_envs, links_names, joints_names, contacts_names=(), xfrc_names=(),
                 animat_options=None, arena_options=None, units=None, buffer_size=1, device=0,
                 team_lanes=0, library=None, log_stride=1):
        # pylint: disable=too-many-arguments,too-many-locals
        self.lib = load_library(library)
        self.model = model
        self.n_envs = int(n_envs)
        self.buffer_size = int(buffer_size)
        # Physics steps per logged iteration (num_sub_steps x n_sub_steps of the reference's loop,
        # task.py:168-186, 348-369).  The device writes a row after every physics step into a ring
        # of buffer_size*log_stride rows; the reference's row `i` (the state at the full step of
        # iteration i) is device row i*log_stride, which is what the accessors below return.
        self.log_stride = max(1, int(log_stride))
        self.device_ring = self.buffer_size*self.log_stride
        self.units = units if units is not None else SimulationUnitScaling()
        names = AnimatData.from_sensors_names(
            timestep=model.timestep, buffer_size=1, links=list(links_names),
            joints=list(joints_names), contacts=list(contacts_names), xfrc=list(xfrc_names))
        self.names = names.sensors
        self.maps = {'sensors': get_sensor_maps(model)}
        get_physics2data_maps(model, self.names, self.maps['sensors'])
        self.tables = FarmsTables(model, self.names, self.maps['sensors'], animat_options,
                                  arena_options, self.units)
        self._cmodel = cabi.model_to_c(model)
        self._cfarms = cabi.farms_to_c(self.tables)
        handle = _H()
        self._handle = None
        self._check(self.lib.fb_create(self._cmodel.byref(), self._cfarms.byref(), self.n_envs,
                                       int(device), self.device_ring, int(team_lanes),
                                       ct.byref(handle)))
        self._handle = handle
        self._cpg_n_osc = 0
        self._geom_friction = None      # set_env_params(geom_friction=...) as last set
        self._log = cabi.FbLogView()
        self._state = cabi.FbStateView()
        self._derived = cabi.FbDerivedView()
        self._check(self.lib.fb_log_view(handle, ct.byref(self._log)))
        self._check(self.lib.fb_state_view(handle, ct.byref(self._state)))
        self._check(self.lib.fb_derived_view(handle, ct.byref(self._derived)))
        self.iteration = 0

    @classmethod
    def from_spec(cls, spec, n_envs, buffer_size=1, frictionless_pairs='refuse', **kwargs):
        """Build from an ``AnimatSpec`` (models.py): MJCF text + option objects.
        ``frictionless_pairs``: see ``mjcf_subset.parse_mjcf``."""
        model = parse_mjcf(spec.mjcf, frictionless_pairs=frictionless_pairs)
        return cls(model, n_envs, spec.links_names, spec.joints_names, spec.contacts_names,
                   spec.xfrc_names, animat_options=spec.animat_options,
                   arena_options=spec.arena_options, units=spec.simulation_options.units,
                   buffer_size=buffer_size, **kwargs)

    # ------------------------------------------------------------------ utils
    def _check(self, code):
        if code != 0:
            raise EngineError(self.lib.fb_last_error().decode())

    def close(self):
        if self._handle is not None:
            self.lib.fb_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass

    def _read(self, ptr, shape, dtype=np.float32):
        out = np.empty(shape, dtype=dtype)
        self._check(self.lib.fb_copy_to_host(self._handle, _ptr(ptr), out.ctypes.data, out.nbytes))
        return out

    def _write(self, ptr, values, dtype=np.float32):
        arr = np.ascontiguousarray(values, dtype=dtype)
        self._check(self.lib.fb_copy_to_device(self._handle, _ptr(ptr), arr.ctypes.data, arr.nbytes))

    def device_array(self, ptr, shape, typestr='<f4'):
        """Zero-copy view for ``torch.as_tensor(..., device='cuda')`` / cupy."""
        return _DeviceArray(_ptr(ptr), shape, typestr, self)

    # ------------------------------------------------------------ state I/O
    def reset(self, qpos=None, qvel=None):
        """``physics.reset(keyframe_id=0)`` + the reset's ``mj_forward`` (task.py:137)."""
        qp = None if qpos is None else np.ascontiguousarray(qpos, dtype=np.float64)
        qv = None if qvel is None else np.ascontiguousarray(qvel, dtype=np.float64)
        if qp is not None:
            assert qp.shape == (self.n_envs, self.model.nq), qp.shape
        if qv is not None:
            assert qv.shape == (self.n_envs, self.model.nv), qv.shape
        self._check(self.lib.fb_reset(
            self._handle,
            None if qp is None else qp.ctypes.data_as(cabi.c_double_p),
            None if qv is None else qv.ctypes.data_as(cabi.c_double_p)))
        self.iteration = 0

    def reset_envs(self, envs, qpos=None, qvel=None):
        """Restart some environments while the others keep running (fb_reset_envs): each one takes
        its row of ``qpos`` / ``qvel`` (``None``: the keyframe), ctrl 0, and from here on steps as the
        same environment of a freshly reset batch; its episode starts at the current ``iteration``
        (``episode_start``), and its log accessors (``export_farms``, ``log_arrays(env=)``) return
        that episode.  ``self.iteration`` stays the batch counter.

        ``envs``: host int indices (``qpos [len(envs), nq]``, ``qvel [len(envs), nv]``) or a bool
        ``[n_envs]`` host array (rows ``[n_envs, ...]``, those of unmasked environments ignored); or a
        bool / uint8 ``[n_envs]`` CUDA array (``__cuda_array_interface__`` or ``data_ptr()``) with
        float32 CUDA ``qpos [n_envs, nq]`` / ``qvel [n_envs, nv]``: stream-ordered on the engine's
        stream (``fb_device_ptr_stream``), no host synchronisation, and not validated (a non-finite
        row shows as ``flags`` bit 0 after the next step).  Refused between the sub-steps of a
        logged iteration (``iteration % log_stride != 0``)."""
        if self.iteration % self.log_stride:
            raise ValueError(f'reset_envs: iteration {self.iteration} is not a full step (log_stride '
                             f'{self.log_stride}); restart environments between logged iterations')
        if _device_address(envs) is not None:
            self._reset_envs_where(envs, qpos, qvel)
            return
        arr = np.asarray(envs)
        if arr.dtype == np.bool_:
            if arr.shape != (self.n_envs,):
                raise ValueError(f'reset_envs: a bool mask must be [{self.n_envs}], got {list(arr.shape)}')
            idx = np.flatnonzero(arr)
            pick = lambda rows: None if rows is None else np.asarray(rows, dtype=np.float64)[idx]
            qpos, qvel = pick(qpos), pick(qvel)
        else:
            if arr.size and not np.issubdtype(arr.dtype, np.integer):
                raise TypeError(f'reset_envs: envs must be integer indices or a bool mask, got {arr.dtype}')
            idx = arr.reshape(-1)
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        rows = []
        for name, values, width in (('qpos', qpos, self.model.nq), ('qvel', qvel, self.model.nv)):
            if values is None:
                rows.append(None)
                continue
            values = np.ascontiguousarray(values, dtype=np.float64)
            if values.shape != (len(idx), width):
                raise ValueError(f'reset_envs: {name} must be [{len(idx)}, {width}], got {list(values.shape)}')
            rows.append(values)
        self._check(self.lib.fb_reset_envs(
            self._handle, len(idx), idx.ctypes.data_as(ct.POINTER(ct.c_int32)),
            *[None if r is None else r.ctypes.data_as(cabi.c_double_p) for r in rows]))

    def _reset_envs_where(self, mask, qpos, qvel):
        """fb_reset_envs_where on device arrays (no host synchronisation)."""
        shape, typestr = _device_shape(mask)
        if shape != (self.n_envs,) or typestr not in ('|b1', '|u1'):
            raise ValueError(f'reset_envs: a device mask must be bool / uint8 [{self.n_envs}], got {typestr} {list(shape)}')
        ptrs = []
        for name, values, width in (('qpos', qpos, self.model.nq), ('qvel', qvel, self.model.nv)):
            if values is None:
                ptrs.append(None)
                continue
            ptr = _device_address(values)
            if ptr is None:
                raise TypeError(f'reset_envs: with a device mask, {name} must be a CUDA array')
            vshape, vtype = _device_shape(values)
            if vshape != (self.n_envs, width) or vtype != '<f4':
                raise ValueError(f'reset_envs: {name} must be float32 [{self.n_envs}, {width}] on the device, '
                                 f'got {vtype} {list(vshape)}')
            ptrs.append(ptr)
        self._check(self.lib.fb_reset_envs_where(self._handle, _device_address(mask), *ptrs))

    def episode_start(self):
        """int64 ``[n_envs]``: the batch iteration (physics steps since ``reset``) at which each
        environment's current episode began; 0 after ``reset``.  Episode iteration = ``iteration -
        episode_start()``."""
        out = np.zeros(self.n_envs, dtype=np.int64)
        self._check(self.lib.fb_get_episode_start(self._handle, out.ctypes.data_as(cabi.c_int64_p)))
        return out

    def step(self, n_steps=1, want_derived=False, sync=True):
        """``n_steps`` x (control -> mj_step -> log row -> drag) for every environment."""
        self._check(self.lib.fb_step(self._handle, int(n_steps), int(bool(want_derived)),
                                     int(bool(sync))))
        self.iteration += int(n_steps)

    def synchronize(self):
        self._check(self.lib.fb_synchronize(self._handle))

    def last_step_ms(self):
        ms = ct.c_float()
        self._check(self.lib.fb_last_step_ms(self._handle, ct.byref(ms)))
        return float(ms.value)

    def launch_count(self):
        return int(self.lib.fb_launch_count(self._handle))

    def set_ctrl(self, ctrl):
        arr = np.ascontiguousarray(ctrl, dtype=np.float64)
        assert arr.shape == (self.n_envs, self.model.nu), arr.shape
        self._check(self.lib.fb_set_ctrl(self._handle, arr.ctypes.data_as(cabi.c_double_p)))

    def set_ctrl_sequence(self, ctrl):
        """Open-loop control of the next ``K`` steps: ``ctrl[K, n_envs, nu]`` (``None``: off)."""
        if ctrl is None:
            self._check(self.lib.fb_set_ctrl_sequence(self._handle, None, 0))
            return
        arr = np.ascontiguousarray(ctrl, dtype=np.float32)
        assert arr.ndim == 3 and arr.shape[1:] == (self.n_envs, self.model.nu), arr.shape
        self._check(self.lib.fb_set_ctrl_sequence(self._handle, arr.ctypes.data, arr.shape[0]))

    def set_qpos_spring(self, qpos_spring):
        arr = np.ascontiguousarray(qpos_spring, dtype=np.float64)
        assert arr.shape == (self.n_envs, self.model.nq), arr.shape
        self._check(self.lib.fb_set_qpos_spring(self._handle, arr.ctypes.data_as(cabi.c_double_p)))

    def set_env_phase(self, phase):
        arr = np.ascontiguousarray(phase, dtype=np.float64)
        assert arr.shape == (self.n_envs,), arr.shape
        self._check(self.lib.fb_set_env_phase(self._handle, arr.ctypes.data_as(cabi.c_double_p)))

    def set_wave_controller(self, actuators, amplitude, frequency, phase_lag, offset=None):
        """On-device travelling-wave position control (include/farms_b200.h FbWaveController)."""
        if actuators is None or len(actuators) == 0:
            self._check(self.lib.fb_set_wave_controller(self._handle, None))
            return
        n = len(actuators)
        keep = cabi.Marshalled(cabi.FbWaveController())
        keep.struct.n = n
        keep.set_int('actuator', actuators)
        keep.set_double('amplitude', amplitude)
        keep.set_double('frequency', frequency)
        keep.set_double('phase_lag', phase_lag)
        keep.set_double('offset', np.zeros(n) if offset is None else offset)
        self._check(self.lib.fb_set_wave_controller(self._handle, keep.byref()))

    def set_cpg(self, network):
        """On-device CPG (include/farms_b200.h FbCpgNetwork): ``network`` is a dict with the
        struct's array fields (``frequency, amplitude, rate, coupling_from, coupling_to,
        coupling_weight, coupling_bias, out_actuator, out_osc_a, out_osc_b, out_gain,
        out_offset``), or None to switch it off.  Optional ``spring_qpos_adr, spring_osc_a,
        spring_osc_b, spring_gain, spring_offset``: spring references the network drives
        (fb_set_cpg_springrefs; task.py:338-346)."""
        if network is None:
            self._check(self.lib.fb_set_cpg(self._handle, None))
            self._cpg_n_osc = 0
            return
        keep = cabi.Marshalled(cabi.FbCpgNetwork())
        s = keep.struct
        s.n_osc, s.n_coupling, s.n_out = (len(network['frequency']), len(network['coupling_from']),
                                          len(network['out_actuator']))
        for name in ('frequency', 'amplitude', 'rate', 'coupling_weight', 'coupling_bias', 'out_gain', 'out_offset'):
            keep.set_double(name, network[name])
        for name in ('coupling_from', 'coupling_to', 'out_actuator', 'out_osc_a', 'out_osc_b'):
            keep.set_int(name, network[name])
        self._check(self.lib.fb_set_cpg(self._handle, keep.byref()))
        self._cpg_n_osc = int(s.n_osc)
        adr = np.ascontiguousarray(network.get('spring_qpos_adr', ()), dtype=np.int32)
        if len(adr):
            ints = [np.ascontiguousarray(network[k], dtype=np.int32) for k in ('spring_osc_a', 'spring_osc_b')]
            dbl = [np.ascontiguousarray(network[k], dtype=np.float64) for k in ('spring_gain', 'spring_offset')]
            i32 = ct.POINTER(ct.c_int32)
            self._check(self.lib.fb_set_cpg_springrefs(
                self._handle, len(adr), adr.ctypes.data_as(i32), ints[0].ctypes.data_as(i32), ints[1].ctypes.data_as(i32),
                dbl[0].ctypes.data_as(cabi.c_double_p), dbl[1].ctypes.data_as(cabi.c_double_p)))

    def set_cpg_state(self, phase, amplitude=None):
        """Oscillator phases (and amplitudes) ``[n_envs, n_osc]`` of the on-device CPG."""
        ph = np.ascontiguousarray(np.broadcast_to(phase, (self.n_envs, self._cpg_n_osc)), dtype=np.float64)
        am = None if amplitude is None else np.ascontiguousarray(
            np.broadcast_to(amplitude, (self.n_envs, self._cpg_n_osc)), dtype=np.float64)
        self._check(self.lib.fb_set_cpg_state(
            self._handle, ph.ctypes.data_as(cabi.c_double_p),
            am.ctypes.data_as(cabi.c_double_p) if am is not None else None))

    def cpg_state(self):
        """(phase, amplitude) ``[n_envs, n_osc]`` float64 host copies."""
        ph = np.zeros((self.n_envs, self._cpg_n_osc))
        am = np.zeros_like(ph)
        self._check(self.lib.fb_get_cpg_state(self._handle, ph.ctypes.data_as(cabi.c_double_p),
                                              am.ctypes.data_as(cabi.c_double_p)))
        return ph, am

    def set_actuator_forcerange(self, actuators, limited, forcerange):
        """``physics.named.model.actuator_forcelimited / actuator_forcerange`` edits of
        ``initialize_control`` (task.py:274-286); also applied to ``self.model``."""
        acts = np.ascontiguousarray(actuators, dtype=np.int32)
        lim = np.ascontiguousarray(np.broadcast_to(limited, acts.shape), dtype=np.int32)
        rng = np.ascontiguousarray(np.broadcast_to(forcerange, acts.shape + (2,)), dtype=np.float64)
        self._check(self.lib.fb_set_actuator_forcerange(
            self._handle, len(acts), acts.ctypes.data_as(ct.POINTER(ct.c_int32)),
            lim.ctypes.data_as(ct.POINTER(ct.c_int32)), rng.ctypes.data_as(cabi.c_double_p)))
        self.model.actuator_forcelimited = np.array(self.model.actuator_forcelimited).copy()
        self.model.actuator_forcerange = np.array(self.model.actuator_forcerange, dtype=float).reshape(-1, 2).copy()
        self.model.actuator_forcelimited[acts] = lim
        self.model.actuator_forcerange[acts] = rng

    def set_water_velocity(self, velocity):
        self._check(self.lib.fb_set_water_velocity(self._handle, *[float(v) for v in velocity]))

    def set_swimming(self, drag, buoyancy):
        self._check(self.lib.fb_set_swimming(self._handle, int(bool(drag)), int(bool(buoyancy))))

    # fb_set_env_param fields (include/farms_b200.h FB_ENV_*): keyword -> (field, shape of one environment).
    # geom_friction is given per geom and set per collision candidate (FB_ENV_CAND_FRICTION).
    def _env_param_fields(self):
        n_swim = len(self.tables.swim_links_index)
        return {'jnt_stiffness': (0, (self.model.njnt,)), 'dof_damping': (1, (self.model.nv,)),
                'drag_coefficients': (2, (n_swim, 2, 3)), 'water_velocity': (3, (3,)),
                'geom_friction': (4, (self.model.ngeom,)),
                'actuator_gainprm': (5, (self.model.nu,)), 'actuator_biasprm': (6, (self.model.nu, 3))}

    def set_env_params(self, **fields):
        """Per-environment physical parameters (fb_set_env_param): ``jnt_stiffness [n_envs, njnt]``,
        ``dof_damping [n_envs, nv]``, ``drag_coefficients [n_envs, n_swim, 2, 3]`` (the layout of
        ``FarmsTables.swim_coefficients``), ``water_velocity [n_envs, 3]`` and ``geom_friction [n_envs,
        ngeom]`` (the sliding friction ``model.geom_friction[:, 0]``; each collision candidate gets the
        two geoms' values mixed as the compiler mixes them, ``mjcf_subset.candidate_friction``, and
        explicit ``<pair>`` candidates keep the pair's friction), ``actuator_gainprm [n_envs, nu]`` (the
        fixed gain ``model.actuator_gainprm[:, 0]``, the only column the step reads) and
        ``actuator_biasprm [n_envs, nu, 3]`` (``model.actuator_biasprm[:, 0:3]``).  A ``<position kp>``
        actuator is gain ``kp`` and bias ``[0, -kp, 0]``, a ``<velocity kv>`` gain ``kv`` and bias
        ``[0, 0, -kv]``: a kp sweep sets ``gainprm[:, a] = kp`` and ``biasprm[:, a, 1] = -kp``.  Gains
        and biases have no sign check (MuJoCo has none); a kv too large for the explicit Euler step
        diverges and shows in ``flags``.  Environment ``e`` then steps as the model edited to its
        values.  Only the keywords passed change; ``None`` returns a field to the model's value; an
        array without the environment axis is broadcast to every environment.  The tables survive
        ``reset`` and ``reset_envs``."""
        known = self._env_param_fields()
        for name in fields:
            if name not in known:
                raise TypeError(f'set_env_params: unknown field {name!r} (one of {", ".join(known)})')
        for name, values in fields.items():
            field, shape = known[name]
            if values is None:
                self._check(self.lib.fb_set_env_param(self._handle, field, None))
                if name == 'geom_friction':
                    self._geom_friction = None
                continue
            arr = np.asarray(values, dtype=np.float64)
            if arr.shape != (self.n_envs,) + shape:
                try:
                    arr = np.broadcast_to(arr, (self.n_envs,) + shape)
                except ValueError:
                    raise ValueError(f'set_env_params: {name} must be {list(shape)} or '
                                     f'{[self.n_envs] + list(shape)}, got {list(arr.shape)}') from None
            arr = np.ascontiguousarray(arr)
            if name == 'geom_friction':
                self._set_geom_friction(arr)
                continue
            self._check(self.lib.fb_set_env_param(self._handle, field, arr.ctypes.data_as(cabi.c_double_p)))

    def _set_geom_friction(self, geom_friction):
        """FB_ENV_CAND_FRICTION from per-geom sliding frictions [n_envs, ngeom]."""
        bad = np.argwhere(~(np.isfinite(geom_friction) & (geom_friction >= 0.0)))
        if len(bad):
            e, g = bad[0]
            raise ValueError(f'set_env_params: geom_friction of environment {e}, geom {g} '
                             f'("{self.model.geom_names[g]}") is {float(geom_friction[e, g])!r}: '
                             'a friction must be finite and non-negative')
        cand = np.ascontiguousarray(candidate_friction(self.model, geom_friction))
        try:
            self._check(self.lib.fb_set_env_param(self._handle, 4, cand.ctypes.data_as(cabi.c_double_p)))
        except EngineError as err:
            pair = np.isin(self.model.cand_end, (20, 21))
            low = np.argwhere((cand < PAIR_MIN_FRICTION) & ~pair)
            if not len(low):
                raise
            e, c = low[0]
            g1, g2 = (self.model.geom_names[g[c]] for g in (self.model.cand_geom1, self.model.cand_geom2))
            raise EngineError(f'set_env_params: geom_friction of environment {e} mixes to {cand[e, c]:g} on '
                              f'candidate {c}, geoms "{g1}" and "{g2}" (the larger of the two, or the '
                              f'higher-priority one, is what counts): {err}') from None
        self._geom_friction = geom_friction.copy()

    def env_params(self):
        """The fields of ``set_env_params`` as float64 ``[n_envs, ...]`` arrays (the model's value
        broadcast for a field that is not set)."""
        out = {}
        for name, (field, shape) in self._env_param_fields().items():
            if name == 'geom_friction':
                out[name] = (self._geom_friction.copy() if self._geom_friction is not None else
                             np.tile(np.asarray(self.model.geom_friction, dtype=np.float64)[:, 0], (self.n_envs, 1)))
                continue
            arr = np.zeros((self.n_envs,) + shape, dtype=np.float64)
            if arr.size:
                self._check(self.lib.fb_get_env_param(self._handle, field, arr.ctypes.data_as(cabi.c_double_p)))
            out[name] = arr
        return out

    # --------------------------------------------------------------- views
    @property
    def qpos_spring(self):
        """``model.qpos_spring`` per environment (task.py:343-346), float64 host copy."""
        return self._read(self._state.qpos_spring_dev, (self.n_envs, self.model.nq)).astype(np.float64)

    @property
    def qpos(self):
        return self._read(self._state.qpos_dev, (self.n_envs, self.model.nq))

    @property
    def qvel(self):
        return self._read(self._state.qvel_dev, (self.n_envs, self.model.nv))

    @property
    def ctrl(self):
        return self._read(self._state.ctrl_dev, (self.n_envs, max(1, self.model.nu)))[:, :self.model.nu]

    @property
    def xfrc_applied(self):
        return self._read(self._state.xfrc_applied_dev, (self.n_envs, self.model.nbody, 6))

    @property
    def flags(self):
        return self._read(self._state.flags_dev, (self.n_envs,), np.int32)

    def set_state(self, qpos=None, qvel=None):
        """Overwrite qpos/qvel without re-running the reset forward pass."""
        if qpos is not None:
            self._write(self._state.qpos_dev, qpos)
        if qvel is not None:
            self._write(self._state.qvel_dev, qvel)

    def derived(self):
        """mjData-like quantities of the state the last step/reset ran forward on."""
        d, n, m = self._derived, self.n_envs, self.model
        mc = int(d.maxcon)
        out = dict(
            xpos=self._read(d.xpos_dev, (n, m.nbody, 3)), xquat=self._read(d.xquat_dev, (n, m.nbody, 4)),
            xipos=self._read(d.xipos_dev, (n, m.nbody, 3)),
            linvel=self._read(d.linvel_dev, (n, m.nbody, 3)),
            angvel=self._read(d.angvel_dev, (n, m.nbody, 3)),
            actuator_force=self._read(d.actuator_force_dev, (n, max(1, m.nu)))[:, :m.nu],
            jnt_limit_force=self._read(d.jnt_limit_force_dev, (n, max(1, m.njnt))),
            qacc=self._read(d.qacc_dev, (n, m.nv)),
            ncon=self._read(d.ncon_dev, (n,), np.int32),
            con_cand=self._read(d.con_cand_dev, (n, mc), np.int32),
            con_dist=self._read(d.con_dist_dev, (n, mc)),
            con_pos=self._read(d.con_pos_dev, (n, mc, 3)),
            con_frame=self._read(d.con_frame_dev, (n, mc, 9)),
            con_force=self._read(d.con_force_dev, (n, mc, 3)),
        )
        return out

    def log_arrays(self, env=None):
        """Host copy of the device log: dict of ``[n_envs, ring, n_items, n_cols]`` float32
        (or ``[ring, n_items, n_cols]`` for one ``env``: exactly the reference's
        ``data.sensors.<kind>.array`` shape, task.py:158).  The whole batch comes in batch rows; one
        ``env`` comes as its current episode (``reset_envs``): row ``i`` of the episode's latest pass
        over the ring, rows the episode has not reached zero."""
        log, names = self._log, self.names
        start = 0 if env is None else int(self.episode_start()[int(env)])
        shapes = dict(
            links=(log.links_dev, len(names.links.names), sc.link_size, log.links_vec),
            joints=(log.joints_dev, len(names.joints.names), sc.joint_size, log.joints_vec),
            contacts=(log.contacts_dev, len(names.contacts.names), sc.contact_size, log.contacts_vec),
            xfrc=(log.xfrc_dev, len(names.xfrc.names), sc.xfrc_size, log.xfrc_vec),
        )
        out = {}
        ring, pad, stride = self.buffer_size, int(log.env_pad), self.log_stride
        for kind, (ptr, n_items, cols, vec) in shapes.items():
            if n_items == 0:
                shape = (self.n_envs, ring, 0, cols)
                out[kind] = np.zeros(shape if env is None else shape[1:], dtype=np.float32)
                continue
            # device layout [ring][items][cols/V][env_pad][V] (include/farms_b200.h, FbLogView)
            raw = self._read(ptr, (ring*stride, n_items, cols//vec, pad, vec))[::stride]
            if env is None:
                arr = raw[:, :, :, :self.n_envs, :].transpose(3, 0, 1, 2, 4)
                out[kind] = np.ascontiguousarray(arr).reshape(self.n_envs, ring, n_items, cols)
            else:
                arr = raw[:, :, :, int(env), :]
                if start > 0:
                    # episode row r is device row (start + r*stride) % (ring*stride), a multiple of the
                    # stride (reset_envs runs at full steps); rows past the episode's latest
                    # iteration were not written in this episode
                    r = np.arange(ring)
                    arr = arr[(start//stride + r) % ring]
                    arr[r*stride > self.iteration - start] = 0.0
                out[kind] = np.ascontiguousarray(arr).reshape(ring, n_items, cols)
        return out

    def log_row(self, kind, index, latest=False):
        """Ring row ``index`` of one log kind for every environment: ``[n_envs, n_items,
        n_cols]`` float32 (what ``physics2data`` wrote into ``data.sensors.<kind>.array
        [index]`` in the reference, physics.py:527-545).  ``latest``: the row of the last physics
        step instead (``index`` ignored) -- what the reference's sensor refresh reads on a
        sub-step, where the row it writes to is not the one the state belongs to."""
        log, names = self._log, self.names
        ptr, n_items, cols, vec = dict(
            links=(log.links_dev, len(names.links.names), sc.link_size, log.links_vec),
            joints=(log.joints_dev, len(names.joints.names), sc.joint_size, log.joints_vec),
            contacts=(log.contacts_dev, len(names.contacts.names), sc.contact_size, log.contacts_vec),
            xfrc=(log.xfrc_dev, len(names.xfrc.names), sc.xfrc_size, log.xfrc_vec),
        )[kind]
        if n_items == 0:
            return np.zeros((self.n_envs, 0, cols), dtype=np.float32)
        pad = int(log.env_pad)
        device_row = self.iteration % self.device_ring if latest else int(index)*self.log_stride
        base = _ptr(ptr) + 4*device_row*n_items*cols*pad
        raw = self._read(base, (n_items, cols//vec, pad, vec))
        arr = raw[:, :, :self.n_envs, :].transpose(2, 0, 1, 3)
        return np.ascontiguousarray(arr).reshape(self.n_envs, n_items, cols)

    def export_farms(self, env, data=None):
        """Fill (or create) a reference-shaped float64 ``AnimatData`` for one environment."""
        names = self.names
        if data is None:
            data = AnimatData.from_sensors_names(
                timestep=self.model.timestep, buffer_size=self.buffer_size,
                links=names.links.names, joints=names.joints.names,
                contacts=names.contacts.names, xfrc=names.xfrc.names)
        if self.log_stride > 1:
            # fb_export_farms writes every device row: export those, keep the full-step rows
            full = AnimatData.from_sensors_names(
                timestep=self.model.timestep, buffer_size=self.device_ring,
                links=names.links.names, joints=names.joints.names,
                contacts=names.contacts.names, xfrc=names.xfrc.names)
            stride, self.log_stride = self.log_stride, 1
            try:
                self.export_farms(env, full)
            finally:
                self.log_stride = stride
            for kind in ('links', 'joints', 'contacts', 'xfrc'):
                getattr(data.sensors, kind).array[...] = getattr(full.sensors, kind).array[::stride]
            return data
        ptrs = []
        for arr in (data.sensors.links.array, data.sensors.joints.array,
                    data.sensors.contacts.array, data.sensors.xfrc.array):
            assert arr.dtype == np.float64 and arr.flags['C_CONTIGUOUS']
            ptrs.append(arr.ctypes.data_as(cabi.c_double_p) if arr.size else None)
        self._check(self.lib.fb_export_farms(self._handle, int(env), *ptrs))
        return data

    def step_host(self, n_steps, ctrl=None, qpos=None, qvel=None, links_row=None, joints_row=None,
                  pipelined=False):
        """End-to-end call on HOST float32 buffers (pinned recommended): upload
        ctrl/qpos/qvel (each optional), step, download the last links/joints log
        row of every environment.  ``pipelined``: return once enqueued; the download overlaps
        the next call's kernels (alternate two or more buffer sets, ``host_wait()`` at the end).
        Returns the call's index for ``host_wait_call`` when rows were asked for."""
        def addr(arr):
            if arr is None:
                return None
            if hasattr(arr, 'data_ptr'):
                return arr.data_ptr()
            return arr.ctypes.data
        fn = self.lib.fb_step_host_async if pipelined else self.lib.fb_step_host
        call = int(self.lib.fb_host_call_count(self._handle))
        self._check(fn(self._handle, addr(ctrl), addr(qpos), addr(qvel),
                       int(n_steps), addr(links_row), addr(joints_row)))
        self.iteration += int(n_steps)
        return call if (links_row is not None or joints_row is not None) else None

    def set_host_joint_columns(self, columns=None):
        """Columns of the joints row ``step_host`` downloads (``joints_row`` is then
        ``[n_envs, n_joints, len(columns)]``); ``None`` = the reference's full row."""
        cols = [] if columns is None else [int(c) for c in columns]
        arr = (ct.c_int32*max(1, len(cols)))(*cols)
        self._check(self.lib.fb_set_host_joint_columns(self._handle, len(cols), arr))

    def set_host_link_columns(self, columns=None):
        """Columns of the links row ``step_host`` downloads (``links_row`` is then
        ``[n_envs, n_links, len(columns)]``); ``None`` = the full 20-column row."""
        cols = [] if columns is None else [int(c) for c in columns]
        arr = (ct.c_int32*max(1, len(cols)))(*cols)
        self._check(self.lib.fb_set_host_link_columns(self._handle, len(cols), arr))

    def set_host_ctrl_columns(self, actuators=None):
        """Actuators the ``ctrl`` argument of ``step_host`` carries (``ctrl`` is then ``[n_envs,
        len(actuators)]``; the other ctrl entries keep their device value); ``None`` = all."""
        idx = [] if actuators is None else [int(i) for i in actuators]
        arr = (ct.c_int32*max(1, len(idx)))(*idx)
        self._check(self.lib.fb_set_host_ctrl_columns(self._handle, len(idx), arr))

    def set_host_link_items(self, items=None):
        """Links whose rows ``step_host`` downloads (``links_row`` is then ``[n_envs, len(items),
        columns]``); ``None`` = every link."""
        idx = [] if items is None else [int(i) for i in items]
        arr = (ct.c_int32*max(1, len(idx)))(*idx)
        self._check(self.lib.fb_set_host_link_items(self._handle, len(idx), arr))

    def export_rows(self, kind, row0, n_rows, out=None):
        """Ring rows ``row0 .. row0+n_rows-1`` (modulo the ring) of one log kind for EVERY
        environment as float32 ``[n_rows, n_envs, n_items, n_cols]`` on the host: the streamed
        full-log export (fb_export_rows).  ``out``: a preallocated (pinned) torch tensor / array
        of that many float32 to fill.  ``out[r, e]`` is the reference's
        ``data.sensors.<kind>.array[row0 + r]`` of environment ``e`` (task.py:158).  Rows are
        device rows: with ``log_stride`` > 1 the reference's row ``i`` is device row
        ``i*log_stride``."""
        names = self.names
        n_items, cols, code = dict(
            links=(len(names.links.names), sc.link_size, 0), joints=(len(names.joints.names), sc.joint_size, 1),
            contacts=(len(names.contacts.names), sc.contact_size, 2), xfrc=(len(names.xfrc.names), sc.xfrc_size, 3))[kind]
        shape = (int(n_rows), self.n_envs, n_items, cols)
        if out is None:
            out = np.empty(shape, dtype=np.float32)
        ptr = out.data_ptr() if hasattr(out, 'data_ptr') else out.ctypes.data
        if n_items:
            self._check(self.lib.fb_export_rows(self._handle, code, int(row0), int(n_rows), ptr))
        return out

    def host_wait_slot(self, slot):
        """Completion of the copies of the latest pipelined call with index % 2 == slot."""
        self._check(self.lib.fb_host_wait_slot(self._handle, int(slot)))

    def host_wait_call(self, call):
        """Completion of the copies of the pipelined ``step_host`` that returned ``call``."""
        self._check(self.lib.fb_host_wait_call(self._handle, int(call)))

    def host_wait(self):
        """Completion of every pipelined ``step_host`` issued so far (fb_host_wait)."""
        self._check(self.lib.fb_host_wait(self._handle))

    # ---------------------------------------------------------- introspection
    @property
    def team_lanes(self):
        return int(self.lib.fb_team_lanes(self._handle))

    def set_fast_path(self, enable):
        """Kernel selection (include/farms_b200.h): ``False`` sends every environment
        to the team kernel; the default runs the environment-per-thread kernel first."""
        self._check(self.lib.fb_set_fast_path(self._handle, int(bool(enable))))

    @property
    def fast_path(self):
        """0 = team kernel only, else environments per block of the per-thread kernel."""
        return int(self.lib.fb_fast_path(self._handle))

    def set_fast_slim(self, enable):
        """Large-batch layout of the unconstrained kernel (include/farms_b200.h): 0 / False =
        regular, else 1 .. 8 warps per block."""
        self._check(self.lib.fb_set_fast_slim(self._handle, int(enable)))

    @property
    def fast_slim(self):
        return int(self.lib.fb_fast_slim(self._handle))

    def set_fast_split(self, enable):
        """Use or not the SPLIT variant of the unconstrained kernel (several warps per 32
        environments, small batches; fb_set_fast_split)."""
        self._check(self.lib.fb_set_fast_split(self._handle, int(bool(enable))))

    @property
    def fast_split(self):
        """Warps per 32 environments when ``step`` launches the SPLIT variant, else 0."""
        return int(self.lib.fb_fast_split(self._handle))

    def set_con_split(self, enable):
        """Use or not the SPLIT variant of the constrained per-thread kernel (fb_set_con_split)."""
        self._check(self.lib.fb_set_con_split(self._handle, int(bool(enable))))

    @property
    def con_split(self):
        """True when the next launch hands fully handed-over groups to the SPLIT constrained kernel."""
        return bool(self.lib.fb_con_split(self._handle))

    def fast_split_schedule(self):
        """The tree split: list (one entry per warp) of (phase A bodies, phase B bodies)."""
        n, bnd = (ct.c_int32*4)(), (ct.c_int32*4)()
        order = (ct.c_uint8*(4*64))()
        nw = int(self.lib.fb_fast_split_schedule(self._handle, n, bnd, order))
        out = []
        for w in range(nw):
            bodies = [int(order[64*w + i]) for i in range(n[w])]
            out.append((bodies[:bnd[w]], bodies[bnd[w]:]))
        return out

    def set_fast_lean(self, enable):
        """Use (default) or not the LEAN variants of the unconstrained kernel (fb_set_fast_lean)."""
        self._check(self.lib.fb_set_fast_lean(self._handle, int(bool(enable))))

    @property
    def fast_lean(self):
        """True when ``step`` launches the LEAN variant for this model."""
        return bool(self.lib.fb_fast_lean(self._handle))

    def set_constraint_path(self, per_thread):
        """Who finishes environments with an active joint limit / plane contact: ``True``
        (default) the per-thread constrained kernel, ``False`` the team kernel."""
        self._check(self.lib.fb_set_constraint_path(self._handle, int(bool(per_thread))))

    @property
    def constraint_path(self):
        """1 = per-thread constrained kernel, 0 = team kernel."""
        return int(self.lib.fb_constraint_path(self._handle))

    @property
    def fast_smem_bytes_per_env(self):
        return int(self.lib.fb_fast_smem_bytes_per_env(self._handle))

    @property
    def last_pending(self):
        """Environments the team kernel had to finish in the last ``step``."""
        count = ct.c_int(0)
        self._check(self.lib.fb_last_pending(self._handle, ct.byref(count)))
        return int(count.value)

    @property
    def smem_bytes_per_env(self):
        return int(self.lib.fb_smem_bytes_per_env(self._handle))

    @property
    def log_view(self):
        return self._log

    @property
    def state_view(self):
        return self._state

    @property
    def log_bytes_per_env_step(self):
        n = self.names
        return 4*(sc.link_size*len(n.links.names) + sc.joint_size*len(n.joints.names)
                  + sc.contact_size*len(n.contacts.names) + sc.xfrc_size*len(n.xfrc.names))
