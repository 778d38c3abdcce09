"""CPU-side checks of the trajectory rollout (mt_rollout, BatchedEnvs.rollout) that need no device.

- The alignment rule of every bulk copy on a trajectory slice (slice_bulk_ok in mt_step.cuh), compiled by nvcc into a
  host program and compared with the plain arithmetic: slice s of rows of `row_bytes` may take a bulk copy exactly
  when s * N * row_bytes is a multiple of 16.
- mt_rollout's argument errors, which it reports before it looks at the handle.
- BatchedEnvs.rollout's shape and dtype checks, which run before the library is called.
"""
import os
import subprocess

import numpy as np
import pytest

from manytor_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = 0x7F3A00000000                           # a 16-byte aligned device-like address
N_VALUES = [8 * 1000 + r for r in range(8)] + [1 << 20]
STEPS = [0, 1, 2, 3, 5, 7, 36, 4100]

PROGRAM = r"""
#include <cstdio>
#include "mt_step.cuh"
int main() {
    const unsigned long long base = %dull;
    const long long ns[] = {%s};
    const long long steps[] = {%s};
    for (long long n : ns)
        for (long long s : steps)
            for (long long row : {0ll, 32ll, 32ll * 1000})
                for (int kind = 0; kind < 3; ++kind)              // 0 fp32 obs, 1 binary16 obs, 2 actions
                    for (int v = 1; v <= (kind == 2 ? 8 : 32); ++v) {
                        if (kind == 2 && v < 2) continue;
                        const unsigned long long rb = kind == 0 ? 12ull * v : kind == 1 ? 6ull * v : 4ull * v;
                        std::printf("%%lld %%lld %%lld %%d %%d %%d %%llu\n", n, s, row, kind, v,
                                    (int)mt::slice_bulk_ok(base, s, n, row, rb), mt::slice_row_addr(base, s, n, row, rb));
                    }
    return 0;
}
"""


def test_slice_bulk_predicate_matches_arithmetic(tmp_path):
    src = tmp_path / "pred.cu"
    src.write_text(PROGRAM % (BASE, ", ".join(map(str, N_VALUES)), ", ".join(map(str, STEPS))))
    exe = str(tmp_path / "pred")
    res = subprocess.run([build.find_nvcc(), "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                          "-I", os.path.join(ROOT, "manytor_b200", "csrc"), str(src), "-o", exe],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lines = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split("\n")
    rows = [tuple(int(v) for v in ln.split()) for ln in lines if ln]
    assert len(rows) == len(N_VALUES) * len(STEPS) * 3 * (32 + 32 + 7)
    seen_bad = {0: 0, 1: 0, 2: 0}
    for n, s, row, kind, v, ok, addr in rows:
        rb = {0: 12 * v, 1: 6 * v, 2: 4 * v}[kind]
        assert addr == BASE + (s * n + row) * rb                  # 64-bit: passes 2^32 at 2^20 envs
        # the plain arithmetic of the rule: fp32 needs s N X % 4 == 0, binary16 s N X % 8 == 0, actions s N J % 4 == 0
        want = (s * n * v) % (8 if kind == 1 else 4) == 0
        assert bool(ok) == want, (n, s, row, kind, v)
        seen_bad[kind] += not ok
        if s == 1:                                                # every slice aligned <=> the first one after 0 is
            assert bool(ok) == ((n * rb) % 16 == 0)
    assert all(seen_bad.values())                                 # the misaligned case occurs for every kind


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


A16, A4 = 0x10000, 0x10004              # never dereferenced: every case fails before the handle is looked at


@pytest.mark.parametrize("args, message", [
    ((-1, A16, None, A16, A16, A16), b"n_steps < 0"),
    ((4, A4, None, A16, A16, A16), b"actions_dev must be 16-byte aligned"),
    ((4, None, A4, A16, A16, A16), b"drawn_dev must be 16-byte aligned"),
    ((4, A16, A16, A16, A16, A16), b"drawn_dev must be NULL when actions_dev is given"),
    ((4, None, None, A4, A16, A16), b"obs_dev must be 16-byte aligned"),
    ((4, None, None, A16, None, A16), b"reward_dev is NULL"),
    ((4, None, None, None, A16, None), b"done_dev is NULL"),
    ((4, None, None, A16, A4, A16), b"reward_dev must be 16-byte aligned"),
    ((4, A16, None, None, A16, A16), b"env is NULL"),
])
def test_mt_rollout_argument_errors(lib, args, message):
    k, act, drawn, obs, rew, done = args
    assert lib.mt_rollout(None, k, act, drawn, obs, rew, done, None) == -1     # MT_ERR_INVALID
    assert message in lib.mt_last_error()


def _envs_without_library(monkeypatch, obs_dtype=None):
    """A BatchedEnvs of 8 envs, X = 10, J = 4 whose library calls fail the test."""
    import torch
    from manytor_b200 import core

    class NoLibrary:
        def __getattr__(self, name):
            raise AssertionError(f"the library was called ({name})")

    def no_load(*a, **k):
        raise AssertionError("the library was loaded")

    monkeypatch.setattr(core._lib, "load", no_load)
    env = object.__new__(core.BatchedEnvs)
    env._h = None
    env._lib = NoLibrary()
    env.n, env.x, env.j = 8, 10, 4
    env.obs_dtype = obs_dtype or torch.float32
    env.device = torch.device("cpu")
    return env


def _traj(k, obs_dtype=None, obs_shape=None, reward_dtype=None, actions=None):
    import torch
    from manytor_b200 import Trajectory
    return Trajectory(torch.zeros(obs_shape or (k, 8, 30), dtype=obs_dtype or torch.float32),
                      torch.zeros((k, 8), dtype=reward_dtype or torch.float32), torch.zeros((k, 8), dtype=torch.uint8),
                      actions)


def test_rollout_checks_run_before_the_library(monkeypatch):
    import torch
    env = _envs_without_library(monkeypatch)
    act = np.zeros((3, 8, 4), np.float32)
    cases = [
        (dict(actions=act, record_actions=True), "cannot be combined with actions"),
        (dict(actions=np.zeros((3, 8, 5), np.float32)), r"actions must have shape \(K, 8, 4\)"),
        (dict(actions=np.zeros((8, 4), np.float32)), r"actions must have shape \(K, 8, 4\)"),
        (dict(actions=act, n_steps=4), "disagrees with the 3 steps"),
        (dict(), "needs actions or n_steps"),
        (dict(n_steps=-2), "n_steps must be >= 0"),
        (dict(actions=act, out=(None, None, None, None)), "out must be a Trajectory"),
        (dict(actions=act, out=_traj(3, obs_dtype=torch.float16)), r"out.obs must have shape \(3, 8, 30\) and dtype torch.float32"),
        (dict(actions=act, out=_traj(3, obs_shape=(3, 8, 29))), "out.obs must have shape"),
        (dict(actions=act, out=_traj(4)), "out.obs must have shape"),
        (dict(actions=act, out=_traj(3, reward_dtype=torch.float64)), "out.reward must have shape"),
        (dict(actions=act, write_obs=False, out=_traj(3)), "out.obs must be None here"),
        (dict(actions=act, out=_traj(3, actions=torch.zeros((3, 8, 4)))), "out.actions must be None here"),
        (dict(n_steps=3, record_actions=True, out=_traj(3)), "out.actions must be a tensor"),
        (dict(n_steps=3, record_actions=True, out=_traj(3, actions=torch.zeros((3, 8, 4), dtype=torch.float16))),
         "out.actions must have shape"),
    ]
    for kw, message in cases:
        with pytest.raises(ValueError, match=message):
            env.rollout(**kw)
    env16 = _envs_without_library(monkeypatch, torch.float16)
    with pytest.raises(ValueError, match=r"out.obs must have shape \(3, 8, 30\) and dtype torch.float16"):
        env16.rollout(act, out=_traj(3))
    # right shapes and dtypes, but not on the handle's device: still refused before the library
    env.device = torch.device("cuda", 0)
    with pytest.raises(ValueError, match="contiguous tensor on cuda:0"):
        env.rollout(act, out=_traj(3))
