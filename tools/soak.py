import os, sys, numpy as np, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from farms_mujoco_b200 import models, mjcf_subset
from farms_mujoco_b200.engine import BatchedPhysics
from farms_mujoco_b200.sharding import synthetic_inputs
from farms_mujoco_b200.models import travelling_wave_parameters
name=sys.argv[1]; n=int(sys.argv[2]); launches=int(sys.argv[3])
spec = models.MODELS[name](); model = mjcf_subset.parse_mjcf(spec.mjcf)
qpos0, qvel0, phase = synthetic_inputs(model, np.arange(n))
ph = BatchedPhysics.from_spec(spec, n, buffer_size=8)
ph.set_env_phase(phase)
joints, amp, freq, lag = travelling_wave_parameters(spec)
acts = [model.actuator_id(f'actuator_position_{j}') for j in joints]
ph.set_wave_controller(acts, amp, freq, lag)
ph.reset(qpos0, qvel0)
t=time.time()
for k in range(launches): ph.step(16, sync=False)
ph.synchronize()
f=ph.flags
print(name, n, 'steps', launches*16, 'sec %.2f'%(time.time()-t), 'nonfinite', int(np.count_nonzero(f&1)), 'solver', int(np.count_nonzero(f&4)), 'slim', ph.fast_slim, 'blk', ph.fast_path, 'con_split', ph.con_split, 'finite state', bool(np.isfinite(ph.qpos).all()), 'max|qvel| %.2f'%np.abs(ph.qvel).max())
