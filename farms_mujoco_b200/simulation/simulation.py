"""Simulation (mirror of farms_mujoco/simulation/simulation.py for the batched engine).

``Simulation`` keeps the reference's constructor arguments, ``iteration``, ``run``,
``iterator``, ``postprocess`` and ``save_mjcf_xml``; it steps ``n_envs`` independent
copies of the model on one B200 instead of one copy on one CPU core.

dm_control is not in this image: the three lines of ``Environment.step`` the reference
relies on (SURVEY.md Appendix B) are restated in ``Simulation.step``: the first call
resets (``initialize_episode``, no physics step), every later call is
``before_step -> physics.step(n_sub_steps) -> after_step`` and non-finite states raise
``PhysicsError`` (simulation.py:157-161).

Fused stepping: when no callback and no host-side controller needs to see every
iteration (no callbacks; no controller, a controller that runs on the device, or a host
controller that declares ``open_loop = True`` and whose next K outputs are uploaded as one
sequence, ``fb_set_ctrl_sequence``) ``run`` advances ``chunk`` iterations per kernel launch
(``fb_step(h, K)``); the device log then holds
exactly the rows the per-iteration loop would have produced, and ``postprocess`` reads
them back.  ``chunk=1`` is the reference's ordering step for step.
"""

import os

import numpy as np
import yaml

from ..hdf5_min import write_hdf5
from ..engine import BatchedPhysics
from ..mjcf_subset import parse_mjcf
from .task import ExperimentTask


class PhysicsError(RuntimeError):
    """Diverged state (dm_control.rl.control.PhysicsError, simulation.py:13,157)"""


def extract_sub_dict(dictionary, keys):
    """Extract sub-dictionary (simulation.py:24-30)"""
    return {key: dictionary.pop(key) for key in keys if key in dictionary}


class Simulation:
    """Simulation (simulation.py:33-213), batched"""
    # pylint: disable=too-many-instance-attributes

    def __init__(self, mjcf_model, base_link, simulation_options, legacy_step=False, **kwargs):
        assert not legacy_step, 'legacy_step (mj_step2/mj_step1) gives wrong contact forces (simulation.py:34-38)'
        self._mjcf_model = mjcf_model
        self.options = simulation_options
        self.pause = not self.options.play
        self.handle_exceptions = kwargs.pop('handle_exceptions', False)
        # frictionless <pair>s (the reference's self-collisions): see mjcf_subset.parse_mjcf
        frictionless_pairs = kwargs.pop('frictionless_pairs', 'refuse')
        engine_kwargs = extract_sub_dict(kwargs, (
            'n_envs', 'links_names', 'joints_names', 'contacts_names', 'xfrc_names', 'arena_options',
            'device', 'team_lanes', 'library', 'qpos0', 'qvel0'))
        env_kwargs = extract_sub_dict(kwargs, ('control_timestep', 'n_sub_steps', 'flat_observation'))
        self.n_sub_steps = int(env_kwargs.get('n_sub_steps', 1) or 1)
        # The device writes a log row after EVERY physics step (fb_device.h: fb_run_env); the
        # reference logs on full steps only (task.py:168-186: row = iteration % buffer_size, the
        # iteration advancing once per `substeps` env.steps of `n_sub_steps` physics steps each).
        # The device ring therefore holds log_stride = substeps*n_sub_steps rows per iteration and
        # the reference's row i is device row i*log_stride (engine.BatchedPhysics.log_stride).
        self.log_stride = self.n_sub_steps*max(1, int(self.options.num_sub_steps or 1))
        self.chunk = int(kwargs.pop('chunk', 0))
        assert self.options.headless, 'the viewer is outside the batched path'
        self._qpos0, self._qvel0 = engine_kwargs.pop('qpos0', None), engine_kwargs.pop('qvel0', None)
        buffer_size = kwargs.get('buffer_size', 0) or self.options.buffer_size or self.options.n_iterations
        kwargs['buffer_size'] = buffer_size
        model = parse_mjcf(mjcf_model, frictionless_pairs=frictionless_pairs) if isinstance(mjcf_model, str) else mjcf_model
        animat_options = kwargs.get('animat_options')
        self.physics = BatchedPhysics(
            model, engine_kwargs.pop('n_envs', 1),
            links_names=engine_kwargs.pop('links_names'), joints_names=engine_kwargs.pop('joints_names'),
            contacts_names=engine_kwargs.pop('contacts_names', ()), xfrc_names=engine_kwargs.pop('xfrc_names', ()),
            animat_options=animat_options, arena_options=engine_kwargs.pop('arena_options', None),
            units=self.options.units, buffer_size=buffer_size, log_stride=self.log_stride, **engine_kwargs)
        if self.n_sub_steps > 1 and len(self.physics.tables.swim_links_index):
            # dm_control runs n_sub_steps physics steps inside one env.step with xfrc_applied held
            # (no before_step in between); the fused drag is recomputed every physics step
            raise NotImplementedError(
                'n_sub_steps > 1 with swimming links: the engine refreshes the drag forces every '
                'physics step, the reference holds them across n_sub_steps; use num_sub_steps')
        self.task = ExperimentTask(
            base_link=base_link,
            n_iterations=self.options.n_iterations,
            timestep=self.options.timestep,
            units=self.options.units,
            substeps=self.options.num_sub_steps,
            restart=False,
            device_control=self.log_stride == 1,
            **kwargs,
        )
        self._reset_next_step = True

    @property
    def iteration(self):
        """Iteration"""
        return self.task.iteration

    @classmethod
    def from_spec(cls, spec, n_envs=1, **kwargs):
        """From an ``AnimatSpec`` (models.py): the MJCF text farms_mujoco's ``setup_mjcf_xml``
        would build plus the option objects.  Stands where ``from_sdf`` stands in the
        reference (simulation.py:96-124); the SDF -> MJCF conversion itself is init-time
        host code outside this path."""
        return cls(
            mjcf_model=spec.mjcf, base_link=spec.base_link, simulation_options=spec.simulation_options,
            animat_options=spec.animat_options, arena_options=spec.arena_options, n_envs=n_envs,
            links_names=spec.links_names, joints_names=spec.joints_names,
            contacts_names=spec.contacts_names, xfrc_names=spec.xfrc_names, **kwargs)

    @classmethod
    def from_sdf(cls, simulation_options, animat_options, arena_options, **kwargs):
        """From SDF (simulation.py:96-124): the MJCF is built from ``animat_options.sdf`` by
        ``sdf_subset.spec_from_sdf``, the part of ``setup_mjcf_xml`` / ``sdf2mjcf``
        (mjcf.py:132-600, 1174-1512) the stepping path can run -- primitive collision shapes,
        revolute / prismatic / fixed joints, frames rotated or not, the flat arena of ``arena_options``;
        anything else (meshes, heightmaps, ball / universal joints, joints without limits) raises
        ``NotImplementedError`` naming the element.  The reference's conversion proper needs
        farms_core's SDF reader, trimesh and dm_control.mjcf, none of which exist here."""
        from ..sdf_subset import spec_from_sdf  # pylint: disable=import-outside-toplevel
        n_envs = kwargs.pop('n_envs', 1)
        spec = spec_from_sdf(simulation_options, animat_options, arena_options,
                             contacts_names=kwargs.pop('contacts_names', None))
        return cls.from_spec(spec, n_envs=n_envs, **kwargs)

    def save_mjcf_xml(self, path, verbose=False):
        """Save simulation to mjcf xml (simulation.py:126-132)"""
        text = self._mjcf_model if isinstance(self._mjcf_model, str) else ''
        if verbose:
            print(text)
        with open(path, 'w+', encoding='utf-8') as xml_file:
            xml_file.write(text)

    # ----------------------------------------------------------- Environment.step
    def _check_physics(self):
        flags = self.physics.flags
        if (flags & 1).any():
            raise PhysicsError(f'non-finite state in environments {np.flatnonzero(flags & 1)[:8].tolist()}')

    def step(self, action=None):
        """dm_control ``Environment.step`` (SURVEY.md Appendix B)"""
        if self._reset_next_step:
            self._reset_next_step = False
            self.task.initialize_episode(self.physics)
            if self._qpos0 is not None or self._qvel0 is not None:
                self.physics.reset(self._qpos0, self._qvel0)
            return
        self.task.before_step(action, self.physics)
        self.physics.step(self.n_sub_steps)
        self._check_physics()
        self.task.after_step(self.physics)
        if self.task.get_termination(self.physics):
            self._reset_next_step = True

    def _can_fuse(self):
        task = self.task
        open_loop = getattr(task.controller, 'open_loop', False)
        return (not task.callbacks and (task.controller is None or task.device_controller or open_loop)
                and task.substeps == 1 and self.n_sub_steps == 1)

    def run(self):
        """Run simulation (simulation.py:134-162): ``sim_iterations`` calls of ``step``, the
        first of which is the reset"""
        n_calls = self.task.sim_iterations
        try:
            self.step()
            done = 1
            chunk = self.chunk if self.chunk > 0 else 64
            while done < n_calls:
                if self._can_fuse() and chunk > 1:
                    # K iterations in one launch: the device writes the K log rows itself
                    k = min(chunk, n_calls - done, self.task.n_iterations - self.task.iteration)
                    assert self.task.iteration + k <= self.task.n_iterations
                    if self.task.controller is not None and not self.task.device_controller:
                        # open-loop host controller: its next k outputs travel as one sequence
                        self.physics.set_ctrl_sequence(self.task.control_sequence(k))
                    self.physics.step(k)
                    self._check_physics()
                    self.task.sim_iteration += k
                    self.task.iteration += k
                    done += k
                else:
                    self.step()
                    done += 1
        except PhysicsError as err:
            if self.handle_exceptions:
                return
            raise err
        self.sync_data()

    def iterator(self, show_progress=True, verbose=True):
        """Run simulation (simulation.py:164-179)"""
        del show_progress, verbose
        # as in the reference, the first env.step (inside the first iteration) is the reset
        for iteration in range(self.task.n_iterations):
            yield iteration
            for _ in range(self.task.substeps):
                self.step()

    def sync_data(self):
        """Device log -> ``task.data`` (every row written so far).  The per-iteration loop fills
        ``task.data`` as it goes; after fused launches this brings the host copy up to date."""
        sensors = self.task.data.sensors
        if self.log_stride > 1:
            # never fused: the loop filled the rows as the reference does (including what its
            # sub-step refreshes leave behind); only the row of the state after the last step
            # is missing, when the buffer still has one
            if self.task.iteration < self.task.n_iterations:
                self.task.update_sensors(self.physics)
            return
        logs = self.physics.log_arrays()
        for kind in ('links', 'joints', 'contacts', 'xfrc'):
            target = getattr(sensors, kind).array
            if target.size:
                target[...] = logs[kind]

    def postprocess(self, iteration, log_path='', plot=False, **kwargs):
        """Postprocessing after simulation (simulation.py:181-213).  The reference writes
        ``simulation.hdf5`` through farms_core's ``AnimatData.to_file`` (a nested dict -> HDF5
        groups); h5py and farms_core are not in this image, so the same arrays go to
        ``simulation.npz`` under the keys of that tree as farms_core lays it out to the best of
        our knowledge (UNVERIFIED, SURVEY.md Appendix C): ``timestep``, ``sensors/<kind>/array``
        (here with a leading environment axis: ``[n_envs, iteration, n_items, n_cols]``) and
        ``sensors/<kind>/names``; the flat ``<kind>`` / ``<kind>_names`` keys of round 1 are kept.
        ``simulation.hdf5`` is written too, by ``hdf5_min.write_hdf5`` (a hand-written subset of the
        HDF5 format, read back by its own reader in the tests and by h5py only where h5py exists:
        treat the .npz as the reference copy until it has been).  Options go to the two YAML files
        as in the reference."""
        del kwargs
        assert not plot, 'plotting is outside the batched path'
        times = np.arange(0, self.task.timestep*self.task.n_iterations, self.task.timestep)[:iteration]
        if log_path:
            os.makedirs(log_path, exist_ok=True)
            self.sync_data()
            sensors = self.task.data.sensors
            payload = {'times': times, 'timestep': self.task.timestep}
            for kind in ('links', 'joints', 'contacts', 'xfrc'):
                arr = getattr(sensors, kind)
                names = np.array([str(n) for n in arr.names])
                payload[kind] = arr.array[:, :iteration]
                payload[f'{kind}_names'] = names
                payload[f'sensors/{kind}/array'] = arr.array[:, :iteration]
                payload[f'sensors/{kind}/names'] = names
            np.savez_compressed(os.path.join(log_path, 'simulation.npz'), **payload)
            # simulation.hdf5 (simulation.py:200-202) through the built-in minimal writer: the same
            # tree as groups / datasets; one environment is written in the reference's shapes
            # ([iteration, n_items, n_cols]), a batch keeps its leading environment axis
            single = self.physics.n_envs == 1
            tree = {'timestep': float(self.task.timestep), 'sensors': {}}
            for kind in ('links', 'joints', 'contacts', 'xfrc'):
                arr = getattr(sensors, kind)
                rows = arr.array[:, :iteration]
                tree['sensors'][kind] = {'array': rows[0] if single else rows, 'names': [str(n) for n in arr.names]}
            write_hdf5(os.path.join(log_path, 'simulation.hdf5'), tree)
            with open(os.path.join(log_path, 'simulation_options.yaml'), 'w', encoding='utf-8') as out:
                yaml.safe_dump(_plain(self.options), out)
            if self.task.animat_options is not None:
                with open(os.path.join(log_path, 'animat_options.yaml'), 'w', encoding='utf-8') as out:
                    yaml.safe_dump(_plain(self.task.animat_options), out)
        return times


def _plain(obj):
    """Dataclass / numpy -> YAML-friendly builtins."""
    import dataclasses  # pylint: disable=import-outside-toplevel
    if dataclasses.is_dataclass(obj):
        return {f.name: _plain(getattr(obj, f.name)) for f in dataclasses.fields(obj)}
    if isinstance(obj, dict):
        return {str(k): _plain(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [_plain(v) for v in obj]
    if isinstance(obj, np.ndarray):
        return obj.tolist()
    if isinstance(obj, (np.floating, np.integer)):
        return obj.item()
    if isinstance(obj, (str, int, float, bool)) or obj is None:
        return obj
    if hasattr(obj, '__dict__'):
        return {k: _plain(v) for k, v in vars(obj).items() if not k.startswith('_')}
    return str(obj)
