"""CPU: the C-ABI library loads and exports every symbol include/hvo_capi.h declares (no compute calls)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, 'include', 'hvo_capi.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(hvo_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol(hvo):
    if not os.path.exists(hvo.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(hvo.LIB_PATH)
    names = _declared()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f'{n} declared in hvo_capi.h but not exported'


def test_python_binding_covers_the_header(hvo):
    assert sorted(hvo.ABI) == _declared()


def test_version_and_error_strings(hvo):
    l = hvo.lib()
    assert b'sm_100a' in l.hvo_version()
    assert isinstance(l.hvo_last_error(), bytes)


_NO_DEVICE = '''
import hvo_b200 as hvo
try:
    n = hvo.device_count()
except hvo.HvoError as e:
    assert e.status == hvo.HVO_ERR_CUDA, e
    n = 0
assert n == 0, n
try:
    hvo.ORBextractor(1000, 1.2, 8, 20, 7, width=640, height=480)
except hvo.HvoError as e:
    assert e.status == hvo.HVO_ERR_CUDA, e
else:
    raise AssertionError('created without a device')
print('ok')
'''


def test_create_fails_loudly_without_a_device():
    """No CPU fallback: on a box without CUDA every create call reports HVO_ERR_CUDA.  Checked in a child process that sees no
    device (CUDA_VISIBLE_DEVICES empty), so that it runs on a box with GPUs as well."""
    r = subprocess.run([sys.executable, '-c', _NO_DEVICE], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == 'ok', r.stdout + r.stderr


def test_argument_validation_needs_no_device(hvo):
    with pytest.raises(hvo.HvoError) as ei:
        hvo.ORBextractor(1000, 1.2, 99, 20, 7, width=640, height=480)
    assert ei.value.status == hvo.HVO_ERR_ARG
