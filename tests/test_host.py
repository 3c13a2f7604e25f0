"""CPU-only checks: the C ABI library loads and exports every declared symbol; host logic; no CPU fallback."""
import os
import re

import numpy as np
import pytest

from qtrunk import NORMAL, q_decode, q_encode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from dsen2_b200 import _capi, build
    build.build()
    lib = _capi.lib()
    header = open(os.path.join(ROOT, 'include', 'dsen2_b200.h')).read()
    declared = set(re.findall(r'\b(dsen2_[a-z0-9_]+)\s*\(', header))
    assert declared, "no declarations parsed"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.dsen2_abi_version() == 3


def test_patch_counts_match_reference_arithmetic():
    from dsen2_b200.patches import patch_counts
    assert patch_counts(300, 300, 64, 4) == (36, 36)        # 600x600 scene, ipynb:167
    assert patch_counts(280, 280, 64, 4) == (36, 25)        # SURVEY fact 5: 11 surplus zero patches
    assert patch_counts(100, 100, 32, 2) == (16, 16)        # 60 m path, ipynb:206
    assert patch_counts(5490, 5490, 64, 4) == (9801, 9801)
    assert patch_counts(1830, 1830, 32, 2) == (4356, 4356)
    with pytest.raises(ValueError):
        patch_counts(10, 10, 8, 4)


def test_argument_errors_are_reported_without_a_gpu():
    from dsen2_b200 import _capi
    lib = _capi.lib()
    assert lib.dsen2_extract_patches(None, 10, 10, 4, 2, 64, 4, 0, 1, 1.0, None, None) == -1
    assert b'null pointer' in lib.dsen2_last_error()
    assert lib.dsen2_conv_relu(None, None, None, 1, 8, 8, 128, None, None) == -1
    assert lib.dsen2_s2model_workspace_bytes(1, 128, 10, 128) >= 128 * 128 * (128 + 3 * 128) * 2
    # the feature size / channel count of the training-step entry points (ABI 3) is checked before anything touches the device
    import ctypes
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(ctypes.byref(buf, 1024 - ctypes.addressof(buf) % 1024), ctypes.c_void_p)      # a non-null, aligned pointer
    assert lib.dsen2_conv_res32(p, p, p, 1, 8, 8, 192, 0.1, p, p, None, None) == -1
    assert b'128 or 256' in lib.dsen2_last_error()
    assert lib.dsen2_conv_relu_bwd(p, p, p, p, 1, 8, 8, 64, p, None) == -1
    assert b'128 or 256' in lib.dsen2_last_error()
    assert lib.dsen2_wgrad_nhwc(p, p, 1, 8, 8, 96, 1.0, p, None, None) == -1
    assert b'128 or 256' in lib.dsen2_last_error()
    assert lib.dsen2_conv_head16_relu(p, p, p, p, 1, 8, 8, 128, p, p, None) == -1
    assert b'256 only' in lib.dsen2_last_error()


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from dsen2_b200 import _capi, imresize, patches, supres
    from dsen2_b200.DSen2Net import s2model
    with pytest.raises(_capi.DSen2Error):
        patches.get_test_patches(np.zeros((128, 128, 4), np.float32), np.zeros((64, 64, 6), np.float32))
    with pytest.raises(_capi.DSen2Error):
        imresize.imresize(np.zeros((8, 8, 2), np.float32), 2)
    m = s2model(((4, None, None), (6, None, None)), 1, 128, seed=0)
    with pytest.raises(_capi.DSen2Error):
        m.predict([np.zeros((1, 4, 32, 32), np.float32), np.zeros((1, 6, 32, 32), np.float32)])
    with pytest.raises(_capi.DSen2Error):
        supres.DSen2_20(np.zeros((128, 128, 4), np.float32), np.zeros((64, 64, 6), np.float32), model=m)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'dsen2_b200')
    for dirpath, _d, files in os.walk(pkg):
        for fn in files:
            if fn.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), fn


def test_s2model_shapes_params_and_weight_roundtrip(tmp_path):
    from dsen2_b200.DSen2Net import s2model
    m20 = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=0)
    assert m20.count_params() == 1789574 and len(m20.layer_shapes) == 14      # SURVEY 2.3
    m60 = s2model(((4, None, None), (6, None, None), (2, None, None)), num_layers=6, feature_size=128, seed=0)
    assert m60.count_params() == 1787266 and m60.out_channels == 2
    v20 = s2model(((4, None, None), (6, None, None)))                          # defaults 32 x 256 (DSen2Net.py:18)
    assert v20.count_params() == 37802246 and len(v20.layer_shapes) == 66
    p = str(tmp_path / 's2_032_lr_1e-04.hdf5')
    m20.save_weights(p)
    other = s2model(((4, None, None), (6, None, None)), num_layers=6, feature_size=128, seed=1)
    other.load_weights(p)
    assert all(np.array_equal(a, b) for a, b in zip(m20.get_weights(), other.get_weights()))
    with pytest.raises(ValueError):
        m60.load_weights(p)                                                    # wrong architecture
    with pytest.raises(OSError):
        m20.load_weights(str(tmp_path / 'missing.hdf5'))


def test_load_full_model_file_layout(tmp_path):
    """Keras full-model saves nest weights under /model_weights next to /optimizer_weights (supres_train.py:195-201);
    non-conv layers appear in layer_names with empty weight_names."""
    from dsen2_b200.DSen2Net import s2model
    from dsen2_b200.hdf5 import write_hdf5
    m = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=2)
    ws = m.get_weights()
    names, tree, attrs = [], {}, {}
    conv_i = 0
    for lname in ['input_1', 'input_2', 'concatenate_1', 'conv2d_7', 'conv2d_8', 'activation_3', 'conv2d_9',
                  'lambda_1', 'add_1', 'conv2d_10', 'add_2']:
        names.append(lname.encode())
        if lname.startswith('conv2d'):
            tree[lname] = {lname: {'kernel:0': ws[2 * conv_i], 'bias:0': ws[2 * conv_i + 1]}}
            attrs['/model_weights/' + lname] = {'weight_names': np.array([(lname + '/kernel:0').encode(),
                                                                          (lname + '/bias:0').encode()])}
            conv_i += 1
        else:
            tree[lname] = {}
            attrs['/model_weights/' + lname] = {'weight_names': np.array([], dtype='S1')}
    attrs['/model_weights'] = {'layer_names': np.array(names), 'backend': np.bytes_(b'tensorflow')}
    p = str(tmp_path / 'full.hdf5')
    write_hdf5(p, {'model_weights': tree, 'optimizer_weights': {'iterations:0': np.array([7], np.int64)}}, attrs)
    m2 = s2model(((4, None, None), (6, None, None)), num_layers=1, feature_size=128, seed=9)
    m2.load_weights(p)
    assert all(np.array_equal(a, b) for a, b in zip(ws, m2.get_weights()))


def _write_mat73(path, arrays, chunk=(1, 128, 128)):
    """A MATLAB v7.3 .mat file laid out the way the shipped scenes are: a 512-byte MATLAB header as HDF5 user block
    (superblock base address 512), and each array a chunked dataset (v1 chunk B-tree) through the shuffle + deflate filters,
    with MATLAB_class attributes.  dsen2_b200.hdf5.write_hdf5 only writes contiguous datasets, so the chunked path of the
    reader is exercised with this file."""
    import itertools
    import struct
    import zlib
    from dsen2_b200 import hdf5 as h
    w = h._Writer()
    w.buf += b"\x00" * 96
    members = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        rank, cs = a.ndim, chunk[-a.ndim:]
        keys = []
        for offs in itertools.product(*[range(0, s, c) for s, c in zip(a.shape, cs)]):
            block = np.zeros(cs, a.dtype)                          # edge chunks are stored whole, zero-padded
            sub = a[tuple(slice(o, o + c) for o, c in zip(offs, cs))]
            block[tuple(slice(0, n) for n in sub.shape)] = sub
            shuffled = np.frombuffer(block.tobytes(), np.uint8).reshape(-1, a.itemsize).T.tobytes()
            raw = zlib.compress(shuffled)
            keys.append((len(raw), offs, w.alloc(raw)))
        node = b"TREE" + struct.pack("<BBHQQ", 1, 0, len(keys), h._UNDEF, h._UNDEF)
        for size, offs, addr in keys:
            node += struct.pack("<II%dQQ" % (rank + 1), size, 0, *offs, 0, addr)
        node += struct.pack("<II%dQ" % (rank + 1), 0, 0, *a.shape, 0)
        btree = w.alloc(node)
        filters = struct.pack("<BB6x", 1, 2) + struct.pack("<HHHHI4x", 2, 0, 1, 1, a.itemsize) + \
            struct.pack("<HHHHI4x", 1, 0, 1, 1, 3)               # shuffle (element size), then deflate (level 3)
        members[name] = w.object_header([
            h._msg(0x01, h._ds_message(a.shape)),
            h._msg(0x03, h._dt_message(a), flags=1),
            h._msg(0x05, struct.pack("<BBBB", 2, 2, 0, 0)),
            h._msg(0x08, struct.pack("<BBBQ%dI" % (rank + 1), 3, 2, rank + 1, btree, *cs, a.itemsize)),
            h._msg(0x0B, filters),
            h._attr_message("MATLAB_class", np.bytes_(b"single")),
        ])
    root = w.group(members, {})
    sb = h._SIG + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0)
    sb += struct.pack("<QQQQ", 512, h._UNDEF, len(w.buf), h._UNDEF) + struct.pack("<QQII16x", 0, root, 0, 0)
    w.buf[:96] = sb
    header = b"MATLAB 7.3 MAT-file, Platform: GLNXA64, Created on: Sat May 27 12:00:00 2017 HDF5 schema 1.00 ."
    with open(path, "wb") as fh:
        fh.write(header.ljust(512, b" ") + bytes(w.buf))


@pytest.fixture
def malmo_mat(malmo, tmp_path):
    """The Malmo scene (tests/golden/scene_malmo_u16.npz) as the reference's data/S2A_MSIL1C_20170527_T33UUB.mat stores it:
    single-precision arrays, transposed to MATLAB's column-major order."""
    path = tmp_path / 'S2A_MSIL1C_20170527_T33UUB.mat'
    _write_mat73(str(path), {k: a.transpose() for k, a in zip(('im10', 'im20', 'im60'), malmo)})
    return path


def test_hdf5_reader_on_mat_fixture_if_reference_present(malmo_mat, fingerprints):
    """The scene read back from a MATLAB v7.3 file has the sha1 of the arrays h5py read from the reference's .mat file."""
    import hashlib
    from dsen2_b200.hdf5 import File
    f = File(str(malmo_mat))
    assert f['im10'].attrs['MATLAB_class'] == b'single'
    for k in ('im10', 'im20', 'im60'):
        a = f[k][()]
        assert a.dtype == np.float32
        assert hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:12] == fingerprints['malmo.' + k]


def test_weight_file_naming_convention():
    from dsen2_b200 import supres
    assert supres.SCALE == 2000 and supres.MDL_PATH == '../models/'
    assert supres.weight_file(False, False).endswith('s2_032_lr_1e-04.hdf5')
    assert supres.weight_file(False, True).endswith('s2_030_lr_1e-05.hdf5')
    assert supres.weight_file(True, False).endswith('s2_033_lr_1e-04.hdf5')
    assert supres.weight_file(True, True).endswith('s2_034_lr_1e-04.hdf5')


def test_demo_readh5_and_rmse(malmo, malmo_mat, capsys):
    """demoDSen2.py:14-35 mirrors: RMSE formula, readh5 on the Malmoe scene as a MATLAB v7.3 file."""
    from dsen2_b200 import demoDSen2
    a = np.arange(12, dtype=np.float32).reshape(3, 4)
    b = a + np.float32(2)
    assert demoDSen2.RMSE(a, b) == 2.0 and 'RMSE: 2.0000' in capsys.readouterr().out
    path = str(malmo_mat.parent) + '/'
    old, demoDSen2.DATA_PATH = demoDSen2.DATA_PATH, path
    try:
        d10, d20, d60 = demoDSen2.readh5('S2A_MSIL1C_20170527_T33UUB.mat', im60=True)
    finally:
        demoDSen2.DATA_PATH = old
    assert d10.shape == (600, 600, 4) and d20.shape == (300, 300, 6) and d60.shape == (100, 100, 2) and d10.dtype == np.float32
    assert all(np.array_equal(x, y) for x, y in zip((d10, d20, d60), malmo))


def test_q_trunk_code_properties():
    """fp16 + 8 bit trunk code (include/dsen2_b200.h): 19 significant bits, unbiased, codes are fixed points."""
    rng = np.random.RandomState(3)
    x = np.concatenate([rng.randn(4096) * s for s in (1e-7, 1e-4, 1e-2, 1.0, 300.0)] +
                       [np.array([0.0, -0.0, 2.0 ** -14, 2.0 ** -24, 1e-9, -1e-9, 1.0, -1.0, 65000.0, 0.99999994,
                                  1.0009765])]).astype(np.float32)
    h, lo = q_encode(x)
    y = q_decode(h, lo)
    assert np.isfinite(y).all()
    big = np.abs(x) >= NORMAL
    assert np.abs(y[big].astype(np.float64) / x[big] - 1).max() < 2.0 ** -18          # 19 significant bits
    assert np.abs(y[~big].astype(np.float64) - x[~big]).max() <= 2.0 ** -24            # subnormal x_hi: absolute
    assert (y[x == 0] == 0).all()
    assert np.abs(h.astype(np.float64) - x)[big].max() <= np.abs(x[big]).max() * 2.0 ** -11   # x_hi is x rounded to fp16
    h2, lo2 = q_encode(y[big])                                                         # codes are fixed points
    assert np.array_equal(h2.view(np.uint16), h[big].view(np.uint16)) and np.array_equal(lo2, lo[big])
    assert abs(np.mean((y[big].astype(np.float64) - x[big]) / x[big])) < 2.0 ** -22    # unbiased
