"""The C-ABI library loads here (no GPU) and exports every symbol include/ogb_sampler.h declares."""

import ctypes
import os
import re

from ogbench_b200 import _native, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'ogb_sampler.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(ogb_[a-z0-9_]+)\s*\(', text)))


def test_header_symbols_exported():
    lib = ctypes.CDLL(build.build())
    names = declared_symbols()
    assert len(names) >= 30
    for name in names:
        assert hasattr(lib, name), f'{name} declared in include/ogb_sampler.h but not exported'


def test_binding_covers_header():
    bound = {name for name, _, _ in _native.SIGNATURES}
    assert bound == set(declared_symbols())


def test_abi_version_and_error_string():
    lib = _native.lib()
    assert lib.ogb_abi_version() == 1
    assert isinstance(lib.ogb_last_error(), bytes)


def test_struct_layouts_match_header():
    """sizeof() of the ctypes mirrors equals what the C compiler sees (guards against drift in _native.py)."""
    import subprocess
    import tempfile

    src = '#include <stdio.h>\n#include "ogb_sampler.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(ogb_field), ' \
          'sizeof(ogb_config), sizeof(ogb_goal_draws), sizeof(ogb_draws), sizeof(ogb_key_info), sizeof(ogb_table_info));return 0;}\n'
    with tempfile.TemporaryDirectory() as tmp:
        c = os.path.join(tmp, 'sz.c')
        open(c, 'w').write(src)
        exe = os.path.join(tmp, 'sz')
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), c, '-o', exe])
        sizes = list(map(int, subprocess.check_output([exe]).split()))
    mirrors = [_native.Field, _native.Config, _native.GoalDraws, _native.Draws, _native.KeyInfo, _native.TableInfo]
    assert sizes == [ctypes.sizeof(m) for m in mirrors]


def test_no_device_fails_loudly():
    """Without a GPU the product path raises; it never falls back to a CPU implementation."""
    import numpy as np
    import pytest

    if _native.device_count() > 0:
        pytest.skip('a GPU is present')
    from ogbench_b200 import Dataset

    ds = Dataset.create(observations=np.zeros((4, 2), np.float32), terminals=np.array([0, 1, 0, 1], np.float32))
    with pytest.raises(_native.NativeError):
        ds.sample(2)
