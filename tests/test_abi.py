"""The C-ABI library: builds for sm_100a, loads, exports every symbol the header declares, and
refuses to compute without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_exports_match_header(built_lib):
    hdr = open(os.path.join(ROOT, 'include', 'soundgen_b200.h')).read()
    declared = set(re.findall(r'\b(sgb_[a-z0-9_]+)\s*\(', hdr))
    from soundgen_beta_b200 import _abi
    assert declared == set(_abi.EXPORTS), declared ^ set(_abi.EXPORTS)
    for name in declared:
        assert hasattr(built_lib, name), name
    assert built_lib.sgb_version() == 200


def test_struct_layouts_match(built_lib):
    import hostsim_util as hu
    from soundgen_beta_b200 import _abi
    L = hu.build()
    assert L.hs_sizeof_syllable() == C.sizeof(_abi.Syllable)
    assert C.sizeof(_abi.Syllable) % 8 == 0 and C.sizeof(_abi.Bout) % 8 == 0
    assert C.sizeof(_abi.Noise) % 8 == 0 and C.sizeof(_abi.Envelope) % 8 == 0


def test_sass_has_tma_and_no_library_fft():
    import subprocess
    so = os.path.join(ROOT, 'soundgen_beta_b200', 'libsoundgen_b200.so')
    sass = subprocess.run(['cuobjdump', '-sass', so], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip('cuobjdump unavailable')
    assert 'UBLKCP' in sass            # cp.async.bulk (TMA) staging in the fused filter
    assert 'UTCHMMA' in sass and 'LDTM' in sass and 'STTM' in sass   # tcgen05.mma / TMEM in the additive synthesis (K1)
    assert 'sm_100a' in sass or 'SM100' in sass.upper() or 'sm_100' in sass
    ldd = subprocess.run(['ldd', so], capture_output=True, text=True).stdout
    assert 'cufft' not in ldd and 'torch' not in ldd


NO_DEVICE_CHECK = '''
import numpy as np
import pytest
import soundgen_beta_b200 as sg
assert sg._abi.load().sgb_device_count() == 0
with pytest.raises(sg.SoundgenError) as ei:
    sg.soundgen(sylLen=300, pitchAnchors=[100, 150], temperature=0)
assert ei.value.code == -2
with pytest.raises(sg.SoundgenError):
    sg.getRolloff([150.0])
with pytest.raises(sg.SoundgenError):
    sg.filter_sound(np.zeros(4000), np.ones(400), 800)
'''


def test_no_cpu_fallback(built_lib):
    # a fresh process with every device hidden, so the no-device path runs on GPU machines too
    import subprocess
    import sys
    code = 'import sys; sys.path.insert(0, %r)\n' % ROOT + NO_DEVICE_CHECK
    r = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'soundgen_beta_b200')
    for f in os.listdir(pkg):
        if f.endswith('.py'):
            src = open(os.path.join(pkg, f)).read()
            assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), f
