"""CPU-side checks of the observation format (mt_config.obs_dtype): the field is laid out the same in ctypes and C,
mt_create refuses values other than MT_OBS_F32 / MT_OBS_F16 before it looks for a device, and BatchedEnvs refuses
any other torch dtype before it calls the library."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from manytor_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


def test_obs_dtype_layout_matches_c(lib, tmp_path):
    cfg = _lib.default_config()
    assert cfg.obs_dtype == _lib.MT_OBS_F32 == 0 and _lib.MT_OBS_F16 == 1
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "manytor_b200.h"\n'
                   'int main(void) { printf("%zu %zu %d %d %d\\n", offsetof(mt_config, obs_dtype), sizeof(mt_config), '
                   'MT_OBS_F32, MT_OBS_F16, MT_ABI_VERSION); return 0; }\n')
    exe = str(tmp_path / "layout")
    res = subprocess.run([gcc, "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    off, size, f32, f16, abi = map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert off == _lib.MtConfig.obs_dtype.offset and size == C.sizeof(_lib.MtConfig) == cfg.struct_size
    assert (f32, f16, abi) == (_lib.MT_OBS_F32, _lib.MT_OBS_F16, _lib.MT_ABI_VERSION)


@pytest.mark.parametrize("value", [2, -1])
def test_create_rejects_unknown_obs_dtype(lib, value):
    cfg = _lib.default_config()
    cfg.obs_dtype = value
    h = C.c_void_p()
    assert lib.mt_create(C.byref(cfg), C.byref(h)) == -1               # MT_ERR_INVALID, with or without a GPU
    assert f"obs_dtype must be MT_OBS_F32 (0) or MT_OBS_F16 (1), not {value}".encode() in lib.mt_last_error()
    assert not h


@pytest.mark.parametrize("dtype", ["bfloat16", "float64", "int16"])
def test_batched_envs_rejects_other_dtypes_before_the_library(dtype, monkeypatch):
    import torch
    import manytor_b200
    from manytor_b200 import core

    def no_library(*a, **k):
        raise AssertionError("the library was called")

    monkeypatch.setattr(core._lib, "load", no_library)
    with pytest.raises(ValueError, match="obs_dtype must be torch.float32 or torch.float16"):
        manytor_b200.BatchedEnvs(8, 10, device=0, obs_dtype=getattr(torch, dtype))
    with pytest.raises(ValueError, match="obs_dtype must be torch.float32 or torch.float16"):
        manytor_b200.ManyTorVectorEnv(8, 10, device=0, obs_dtype=getattr(torch, dtype))
