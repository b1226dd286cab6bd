"""The checkpoint file without a GPU: its payload unpickles without loading the CUDA library, and a file of
another format or C-ABI version is refused before anything is unpickled from its payload."""
import os
import pickle
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from geonomics_b200 import _lib, api, checkpoint  # noqa: E402

PARAMS = os.path.join(HERE, 'data', 'params_small.py')


def _payload():
    import numpy as np
    p = api.read_parameters_file(PARAMS)
    np.random.seed(1)
    land = api._make_landscape(p)
    spp_p = p.comm.species.spp_0
    return dict(land=land, gen_arch=api._make_genomic_architecture(spp_p, land), rng=np.random.get_state())


def test_payload_unpickles_without_the_library(tmp_path):
    path = str(tmp_path / 'm.ckpt')
    checkpoint.write(path, _payload(), _lib.GNX_ABI_VERSION)
    code = ('import sys; sys.path.insert(0, %r)\n'
            'from geonomics_b200 import _lib, checkpoint\n'
            'out = checkpoint.read(%r, _lib.GNX_ABI_VERSION)\n'
            'assert out["gen_arch"].L == 60 and len(out["land"]) == 3 and out["land"]._changer is not None\n'
            'assert _lib._LIB is None\n'
            'assert "libgnxb200" not in open("/proc/self/maps").read()\n' % (ROOT, path))
    subprocess.run([sys.executable, '-c', code], check=True)


def _with_header(path, **header):
    h = dict(magic=checkpoint.MAGIC, format=checkpoint.FORMAT_VERSION, abi=_lib.GNX_ABI_VERSION)
    h.update(header)
    with open(path, 'wb') as f:
        pickle.dump(h, f)
        pickle.dump({'model': None}, f)


@pytest.mark.parametrize('header,match', [(dict(format=checkpoint.FORMAT_VERSION + 1), 'format'),
                                          (dict(abi=_lib.GNX_ABI_VERSION + 1), 'C-ABI'),
                                          (dict(magic='something else'), 'not a geonomics_b200 checkpoint')])
def test_other_versions_are_refused(tmp_path, header, match):
    path = str(tmp_path / 'm.ckpt')
    _with_header(path, **header)
    with pytest.raises(checkpoint.CheckpointError, match=match):
        api.load_model(path)


def test_not_a_pickle_is_refused(tmp_path):
    path = tmp_path / 'm.ckpt'
    path.write_bytes(b'\x00not a checkpoint')
    with pytest.raises(checkpoint.CheckpointError, match='not a geonomics_b200 checkpoint'):
        api.load_model(str(path))


def test_write_replaces_the_file_whole(tmp_path):
    path = str(tmp_path / 'm.ckpt')
    checkpoint.write(path, {'a': 1}, _lib.GNX_ABI_VERSION)
    checkpoint.write(path, {'a': 2}, _lib.GNX_ABI_VERSION)
    assert checkpoint.read(path, _lib.GNX_ABI_VERSION) == {'a': 2}
    assert os.listdir(str(tmp_path)) == ['m.ckpt']
