"""AddressSanitizer pass over the device code compiled for the host (tests/emu harness):
    g++ -O1 -g -std=c++17 -fPIC -shared -fsanitize=address -fno-omit-frame-pointer -DFB_HOST_EMU \
        -x c++ farms_mujoco_b200/csrc/fb_engine.cu -o /tmp/libfb_emu_asan.so
    LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0 python tools/asan_emu.py
Walks every layout / kernel selection (regular and SLIM blocks, per-thread and team constraint
paths, box contacts, fixed base, host row gathers) so that an out-of-bounds index into the
per-environment blocks and scratch regions shows up on the GPU-less box (compute-sanitizer is
closed on the GPU pool)."""
import os, sys, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from conftest import make_case
import variant_models
from farms_mujoco_b200 import mjcf_subset
from farms_mujoco_b200.engine import BatchedPhysics
lib='/tmp/libfb_emu_asan.so'
for name in ('swimmer8','salamander_swim','salamander','centipede'):
    for slim in (0,1):
        for pt in (True, False):
            spec, model, qpos0, qvel0, ctrl = make_case(name, 3)
            ph = BatchedPhysics.from_spec(spec, 3, buffer_size=6, library=lib)
            ph.set_fast_slim(slim); ph.set_constraint_path(pt)
            ph.reset(qpos0, qvel0); ph.set_ctrl(ctrl); ph.step(5)
            links=np.zeros((3,len(spec.links_names),20),dtype=np.float32); joints=np.zeros((3,len(spec.joints_names),18),dtype=np.float32)
            ph.step_host(2, ctrl=ctrl.astype(np.float32), links_row=links, joints_row=joints)
            ph.set_host_joint_columns([0,1,11,16]); j4=np.zeros((3,len(spec.joints_names),4),dtype=np.float32)
            ph.step_host(2, ctrl=ctrl.astype(np.float32), links_row=links, joints_row=j4)
            del ph
    print(name,'ok')
spec=variant_models.salamander_box_feet(); model=mjcf_subset.parse_mjcf(spec.mjcf)
ph=BatchedPhysics.from_spec(spec,2,buffer_size=6,library=lib); ph.step(5); print('box ok')
spec=variant_models.swimmer8_fixed_base(); ph=BatchedPhysics.from_spec(spec,2,buffer_size=6,library=lib); ph.step(5); print('fixed ok')
# explicit <pair> self-collisions: the dense Newton Hessian behind the contact Jacobians
from test_emu_parity import _pair_case
spec, model, qpos0, qvel0, ctrl = _pair_case(3)
ph = BatchedPhysics.from_spec(spec, 3, buffer_size=6, library=lib)
ph.reset(qpos0, qvel0); ph.set_ctrl(ctrl); ph.step(5); assert ph.log_arrays()['contacts'].any(); print('pairs ok')
# frictionless pairs as hard normal rows (the working-set regions), alone and beside a mu = 0.5 pair
from test_frictionless_pairs import _case
for kind in ('pair', 'ground', 'mixed'):
    spec, model, qpos0, qvel0, ctrl, _ = _case(kind, 3)
    ph = BatchedPhysics.from_spec(spec, 3, buffer_size=6, library=lib, frictionless_pairs='hard')
    ph.reset(qpos0, qvel0); ph.set_ctrl(ctrl); ph.step(5); assert ph.log_arrays()['contacts'].any() and not ph.flags.any()
    print('frictionless pairs', kind, 'ok')
# the stand-alone drag operator
from drag_cases import check_operator
print('drag operator', check_operator(lib, n=33))
