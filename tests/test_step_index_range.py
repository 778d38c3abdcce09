"""CPU-side checks of the step index's range: MT_STEP_INDEX_MAX is the same in C and in the binding, and
BatchedEnvs.step_index refuses values outside [0, MT_STEP_INDEX_MAX] before it calls the library (it used to store
them modulo 2^64).  The library's own refusal is checked on the GPU (tests/test_gpu_launch_bookkeeping.py)."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from manytor_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_step_index_max_matches_c(tmp_path):
    assert _lib.MT_STEP_INDEX_MAX == 1 << 62
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "limit.c"
    src.write_text('#include <stdio.h>\n#include "manytor_b200.h"\n'
                   'int main(void) { printf("%llu\\n", (unsigned long long)MT_STEP_INDEX_MAX); return 0; }\n')
    exe = str(tmp_path / "limit")
    res = subprocess.run([gcc, "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    assert int(subprocess.run([exe], capture_output=True, text=True, check=True).stdout) == _lib.MT_STEP_INDEX_MAX


class RecordingLibrary:
    def __init__(self):
        self.calls = []

    def mt_set_step_index(self, handle, value):
        self.calls.append(value)
        return 0


def _detached_envs(lib):
    from manytor_b200 import BatchedEnvs
    env = object.__new__(BatchedEnvs)             # no device: only the setter's own logic runs
    env._lib = lib
    env._h = C.c_void_p()
    return env


@pytest.mark.parametrize("value", [-1, -(1 << 64), (1 << 62) + 1, 1 << 63, (1 << 64) - 1, 1 << 64])
def test_setter_refuses_values_outside_the_range(value):
    lib = RecordingLibrary()
    env = _detached_envs(lib)
    with pytest.raises(ValueError, match=r"step_index must be in \[0, 2\*\*62\]"):
        env.step_index = value
    assert lib.calls == []


@pytest.mark.parametrize("value", [0, 1, (1 << 32) + 5, 1 << 62])
def test_setter_passes_values_in_the_range_unchanged(value):
    lib = RecordingLibrary()
    env = _detached_envs(lib)
    env.step_index = value
    assert lib.calls == [value]
