"""The C-ABI library builds, loads and exports every symbol include/vr_b200.h declares; the ctypes table
in lib/_native.py covers exactly that set.  No compute calls (there is no GPU in this container)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from conftest import PKG, ROOT


def _declared():
    src = open(os.path.join(ROOT, 'include', 'vr_b200.h')).read()
    return sorted(set(re.findall(r'VR_API\s+[\w\s\*]+?\b(vr_[a-z0-9_]+)\s*\(', src)))


def test_header_declares_the_surface():
    names = _declared()
    for required in ('vr_create', 'vr_destroy', 'vr_last_error', 'vr_load_tensor', 'vr_finalize_weights', 'vr_stft',
                     'vr_istft', 'vr_predict_mask', 'vr_forward', 'vr_separate', 'vr_separate_windows',
                     'vr_apply_mask', 'vr_apply_mask_istft', 'vr_separate_wave', 'vr_separate_wave_host'):
        assert required in names


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    from lib import _native
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in _declared():
        assert hasattr(lib, name), name
    assert sorted(_native.SIGNATURES) == _declared()


def test_create_fails_loudly_without_gpu():
    """Run in a child process that sees no CUDA device, so that it checks the same thing on a GPU machine."""
    code = ('import pytest\nfrom lib import _native\nwith pytest.raises(_native.NativeError):\n'
            '    _native.Context(0, 2048, 1024, 32, 128, 256, 1)\n')
    r = subprocess.run([sys.executable, '-c', code], cwd=PKG, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_library_missing_is_an_error(monkeypatch, tmp_path):
    from lib import _native
    monkeypatch.setattr(_native, '_lib', None)
    monkeypatch.setattr(_native, 'LIB_PATH', str(tmp_path / 'nope.so'))
    with pytest.raises(ImportError):
        _native.load_library()
