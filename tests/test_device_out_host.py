"""Device output without a device: argument refusals that need no GPU, and the no-device path of the new entry
points (no host fallback: they fail with SGB_ERR_CUDA)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_unsupported_dtype_is_refused_before_device_work(built_lib, monkeypatch):
    torch = pytest.importorskip('torch')
    import soundgen_beta_b200 as sg
    from soundgen_beta_b200 import api

    def no_device_work(*a, **k):
        raise AssertionError('device work before the dtype check')
    monkeypatch.setattr(api, 'FrontEnd', no_device_work)
    monkeypatch.setattr(api, 'Batch', no_device_work)
    for dt in (torch.bfloat16, torch.float16, torch.float64, torch.int32, np.float32, 'f32'):
        with pytest.raises(ValueError):
            sg.soundgen_batch_device([dict(sylLen=100, temperature=0)], dtype=dt)


def test_device_out_struct_mirror(built_lib):
    import ctypes as C
    from soundgen_beta_b200 import _abi
    sizes = (C.c_int32 * 10)()
    assert built_lib.sgb_abi_sizes(sizes, 10) == 0
    assert sizes[9] == C.sizeof(_abi.DeviceOut) == 56
    short = (C.c_int32 * 9)()                      # callers that know nine structs keep working
    assert built_lib.sgb_abi_sizes(short, 9) == 0 and list(short) == list(sizes)[:9]


NO_DEVICE_CHECK = '''
import ctypes as C
import numpy as np
import pytest
import torch
import soundgen_beta_b200 as sg
from soundgen_beta_b200 import _abi
L = _abi.load()
assert L.sgb_device_count() == 0
o = _abi.DeviceOut()
o.dst_elems, o.format = 4, _abi.SGB_OUT_PCM16
off, ln = np.zeros(1, dtype=np.int64), np.full(1, 4, dtype=np.int64)
o.dst_off, o.cap = off.ctypes.data, ln.ctypes.data
buf = np.zeros(4, dtype=np.float32)
assert L.sgb_rows_export(0, buf.ctypes.data, off.ctypes.data, ln.ctypes.data, 1, C.byref(o)) == _abi.SGB_ERR_CUDA
with pytest.raises(sg.SoundgenError) as ei:
    sg.soundgen_batch_device([dict(sylLen=100, pitchAnchors=[100, 150], temperature=0)])
assert ei.value.code == -2
with pytest.raises(sg.SoundgenError) as ei:
    sg.soundgen_batch_device([dict(sylLen=100, pitchAnchors=[100, 150], temperature=0)], dtype=torch.int16)
assert ei.value.code == -2
'''


def test_no_device_path(built_lib):
    pytest.importorskip('torch')
    code = 'import sys; sys.path.insert(0, %r)\n' % ROOT + NO_DEVICE_CHECK
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
