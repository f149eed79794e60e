"""The minimal HDF5 writer behind ``Simulation.postprocess`` (farms_mujoco_b200/hdf5_min.py):
round trip through its own reader (structure: superblock, group B-tree / symbol-table node /
local heap, dataset messages) and, wherever h5py is importable, through libhdf5."""

import os
import struct

import numpy as np
import pytest

from farms_mujoco_b200.hdf5_min import write_hdf5, read_hdf5, SIGNATURE


def _tree():
    rng = np.random.default_rng(0)
    return {
        'timestep': 1e-3,
        'sensors': {
            'links': {'array': rng.normal(size=(7, 3, 20)), 'names': ['link_body_0', 'link_leg_0_L_3', 'c']},
            'joints': {'array': rng.normal(size=(7, 2, 18)).astype(np.float32), 'names': ['j0', 'joint_1']},
            'contacts': {'array': np.zeros((7, 0, 12)), 'names': []},
        },
        'counts': np.arange(5, dtype=np.int32),
        'flag': np.uint8(3),
    }


def _compare(tree, back):
    assert sorted(tree) == sorted(back)
    for key, value in tree.items():
        if isinstance(value, dict):
            _compare(value, back[key])
        elif isinstance(value, list):
            assert [b.decode() for b in np.asarray(back[key]).tolist()] == value
        else:
            got = np.asarray(back[key])
            assert got.shape == np.shape(value) and got.dtype == np.asarray(value).dtype
            assert np.array_equal(got, np.asarray(value))


def test_round_trip_and_fixed_structures(tmp_path):
    path = os.path.join(tmp_path, 'log.hdf5')
    tree = _tree()
    write_hdf5(path, tree)
    raw = open(path, 'rb').read()
    assert raw[:8] == SIGNATURE and raw[8] == 0                       # superblock version 0
    assert raw[13] == 8 and raw[14] == 8                             # 8-byte offsets and lengths
    assert struct.unpack_from('<Q', raw, 40)[0] == len(raw)          # end-of-file address
    assert len(raw) % 8 == 0
    root_header, cache_type = struct.unpack_from('<QI', raw, 64)
    assert cache_type == 1 and raw[root_header] == 1                 # cached symbol table; object header v1
    _compare(tree, read_hdf5(path))


def test_postprocess_writes_the_reference_tree(emu_library, tmp_path):
    """simulation.hdf5 next to simulation.npz: timestep and sensors/<kind>/{array, names}; one
    environment is written in the reference's shapes."""
    from farms_mujoco_b200 import models
    from farms_mujoco_b200.simulation.simulation import Simulation
    spec = models.swimmer8(n_iterations=6)
    sim = Simulation.from_spec(spec, n_envs=1, library=emu_library)
    sim.run()
    sim.postprocess(sim.iteration, log_path=str(tmp_path))
    back = read_hdf5(os.path.join(tmp_path, 'simulation.hdf5'))
    assert float(back['timestep']) == spec.simulation_options.timestep
    links = back['sensors']['links']
    assert links['array'].shape == (sim.iteration, 8, 20) and links['array'].dtype == np.float64
    assert np.array_equal(links['array'], sim.task.data.sensors.links.array[0, :sim.iteration])
    assert [n.decode() for n in links['names']] == spec.links_names
    assert back['sensors']['contacts']['array'].shape[0] == sim.iteration


def test_h5py_reads_the_file(tmp_path):
    """The validation this image cannot run: libhdf5 opening the file."""
    h5py = pytest.importorskip('h5py', reason='h5py is not installed: the hand-written HDF5 file is not validated against libhdf5')
    path = os.path.join(tmp_path, 'log.hdf5')
    tree = _tree()
    write_hdf5(path, tree)
    with h5py.File(path, 'r') as f:
        assert sorted(f) == sorted(tree)
        assert np.array_equal(f['sensors/links/array'][...], tree['sensors']['links']['array'])
        assert [n.decode() for n in f['sensors/links/names'][...]] == tree['sensors']['links']['names']
        assert f['timestep'][()] == tree['timestep']
        assert f['sensors/contacts/array'].shape == (7, 0, 12)


def test_structures_match_a_file_written_by_libhdf5():
    """A file written by libhdf5 itself (MATLAB 7.4, HDF5 1.6; tests/golden/testhdf5_7.4_GLNX86.mat,
    a copy of SciPy's test file scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat, BSD licence;
    512-byte user block): its superblock, root symbol-table entry, B-tree node, symbol-table
    node, local heap and IEEE float64 datatype message are laid out as hdf5_min writes them."""
    sample = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'testhdf5_7.4_GLNX86.mat')
    from farms_mujoco_b200.hdf5_min import _datatype, _read_messages
    raw = open(sample, 'rb').read()
    base = raw.find(SIGNATURE)
    assert base == 512 and raw[base + 8] == 0 and raw[base + 13] == 8 and raw[base + 14] == 8
    assert struct.unpack_from('<Q', raw, base + 24)[0] == base                       # base address
    root_header, cache_type = struct.unpack_from('<QI', raw, base + 64)
    btree, heap = (x + base for x in struct.unpack_from('<QQ', raw, base + 80))
    assert cache_type == 1
    assert raw[btree:btree + 4] == b'TREE' and struct.unpack_from('<BBH', raw, btree + 4) == (0, 0, 1)
    key0, child0, key1 = struct.unpack_from('<QQQ', raw, btree + 24)
    assert raw[heap:heap + 4] == b'HEAP' and raw[heap + 4] == 0
    heap_data = struct.unpack_from('<Q', raw, heap + 24)[0] + base
    snod = child0 + base
    assert raw[snod:snod + 4] == b'SNOD' and struct.unpack_from('<BxH', raw, snod + 4) == (1, 1)
    name_offset, header = struct.unpack_from('<QQ', raw, snod + 8)
    assert key0 == 0 and key1 == name_offset
    assert raw[heap_data + name_offset:].startswith(b'testdouble\x00')
    group_messages = dict(_read_messages(raw, root_header + base))
    assert struct.unpack_from('<QQ', group_messages[0x0011], 0) == (btree - base, heap - base)
    messages = dict(_read_messages(raw, header + base))
    assert bytes(messages[0x0003][:20]) == _datatype(np.float64)                     # the float64 datatype, byte for byte
    assert bytes(messages[0x0001][:8]) == struct.pack('<BBB5x', 1, 2, 0)             # dataspace version 1, rank 2
    assert struct.unpack_from('<QQ', messages[0x0001], 8) == (9, 1)
    assert bytes(messages[0x0005]) == bytes([1, 2, 2, 1, 0, 0, 0, 0])                # the fill-value message written here
