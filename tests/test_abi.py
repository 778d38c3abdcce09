"""CPU-side checks of the C-ABI boundary: the library builds, loads, exports every
symbol include/manytor_b200.h declares, the ctypes structs match the C layout, and
-- with no GPU -- every compute entry point fails loudly instead of falling back."""
import ctypes as C
import os
import re

import pytest

import manytor_b200
from manytor_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "manytor_b200.h")


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mt_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_exported_and_bound(lib):
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
        assert n in _lib.SIGNATURES, f"{n} declared in the header but has no ctypes signature"
    assert sorted(_lib.SIGNATURES) == names


def test_struct_layout_matches_c(lib):
    cfg = _lib.default_config()
    assert cfg.struct_size == C.sizeof(_lib.MtConfig)       # mt_config_init wrote sizeof(mt_config)
    assert C.sizeof(_lib.MtStats) == 8 * _lib.MT_STATS_WORDS
    # reference constants (manytor.py:42-48,162,178,216,231)
    assert (cfg.n_joints, cfg.n_obj, cfg.substeps) == (4, 10, 25)
    assert abs(cfg.radius - 51.3) < 1e-6 and cfg.catch_tol == 8.0
    assert (cfg.action_low, cfg.action_high) == (-180, 180)
    assert [round(cfg.dh[i][2], 4) for i in range(4)] == [4.3, 0.0, 24.3, 0.0]
    assert abs(cfg.dh[3][0] - 27.0) < 1e-6
    assert (cfg.obs_frame, cfg.ground_frame_a, cfg.ground_frame_b, cfg.catch_frame) == (3, 3, 4, 4)
    assert cfg.terminate_on_ground == 0 and cfg.auto_reset == 0   # the code's behaviour, SURVEY Q1/Q2


def test_abi_version(lib):
    assert lib.mt_abi_version() == _lib.MT_ABI_VERSION


def test_bad_config_is_rejected(lib):
    cfg = _lib.default_config()
    h = C.c_void_p()
    cfg.struct_size = 4
    assert lib.mt_create(C.byref(cfg), C.byref(h)) == -1
    assert b"ABI mismatch" in lib.mt_last_error()
    cfg = _lib.default_config()
    cfg.n_obj = 33
    assert lib.mt_create(C.byref(cfg), C.byref(h)) == -1
    assert not h
    for J in (1, 9):                                   # the generic chain is built for J = 2 .. MT_MAX_JOINTS
        cfg = _lib.default_config()
        cfg.n_joints = J
        assert lib.mt_create(C.byref(cfg), C.byref(h)) == -1
        assert b"n_joints must be in [2, 8]" in lib.mt_last_error() and not h
    for field in ("obs_frame", "ground_frame_a", "ground_frame_b", "catch_frame"):
        cfg = _lib.default_config()                    # frames 0 .. J exist; J + 1 does not
        setattr(cfg, field, cfg.n_joints + 1)
        assert lib.mt_create(C.byref(cfg), C.byref(h)) == -1
        assert b"frame selector 5 outside [0, 4]" in lib.mt_last_error() and not h


def test_no_gpu_means_loud_failure(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    cfg = _lib.default_config()
    h = C.c_void_p()
    rc = lib.mt_create(C.byref(cfg), C.byref(h))
    assert rc == -3 and b"no CPU fallback" in lib.mt_last_error()     # MT_ERR_NO_DEVICE
    with pytest.raises(manytor_b200.MantorLibraryError):
        manytor_b200.BatchedEnvs(8, 10)
    import manytor_b200.manytor as tor
    with pytest.raises(manytor_b200.MantorLibraryError):
        tor.Environment(10)
    with pytest.raises(manytor_b200.MantorLibraryError):
        tor.fk(4, [30, 45, 60, 90])


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "manytor_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f


def test_library_is_sm100a_with_tma(lib):
    """The shipped cubin targets sm_100a and the step kernel moves its tiles with TMA
    bulk copies (SASS UBLKCP) -- checked with cuobjdump when it is on PATH."""
    import shutil
    import subprocess
    cu = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cu):
        pytest.skip("cuobjdump not available")
    elf = subprocess.run([cu, "-lelf", _lib.library_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in elf
    sass = subprocess.run([cu, "-sass", _lib.library_path()], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass


def _build_c_host(tmp_path, name="c_host"):
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    exe = str(tmp_path / name)
    lib_dir = os.path.dirname(_lib.library_path())
    cmd = [gcc, "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", name + ".c"),
           "-o", exe, "-L", lib_dir, "-lmanytor_b200", f"-Wl,-rpath,{lib_dir}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_plain_c_host_links_against_the_abi(lib, tmp_path):
    """examples/c_host.c: a host with no CUDA/torch/Python dependency compiles against the header
    (-Wall -Werror) and links the shared library; without a GPU it must fail loudly, not fall back."""
    import subprocess
    import torch
    exe = _build_c_host(tmp_path)
    res = subprocess.run([exe, "64", "2"], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert res.returncode == 0, res.stderr
    else:
        assert res.returncode == 1 and "no CPU fallback" in res.stderr


def test_multi_gpu_c_host_links_against_the_abi(lib, tmp_path):
    """examples/c_host_multi.c (config 4 from plain C: one handle per GPU + mt_stats_allreduce) builds with
    -Wall -Werror against the header; its run is a -m gpu test."""
    _build_c_host(tmp_path, "c_host_multi")


def test_no_prefetch_register_is_overwritten_unread():
    """Regression guard for the hazard that cost 21 % of the step kernel's stall samples: a register that
    receives a tile-ahead prefetch (LDG) must not be written again before something has read it, or the
    overwrite waits for the load and the prefetch becomes a blocking load (tools/sass_waw.py).  Checked
    on the SASS of every reference-arm variant of the built library."""
    import shutil
    import subprocess
    import sys
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from manytor_b200 import _lib
    sass = subprocess.run([cuobjdump, "-sass", _lib.library_path()], capture_output=True, text=True, check=True).stdout
    assert "step_kernelILi0ELi10ELb0ELb1" in sass, "headline kernel missing from the library"
    tool = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "sass_waw.py")
    out = subprocess.run([sys.executable, tool, "step_kernelILi0E"], input=sass, capture_output=True, text=True, check=True).stdout
    assert out.strip().endswith("0 suspicious prefetch overwrite(s)"), out
