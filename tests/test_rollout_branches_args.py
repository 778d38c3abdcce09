"""CPU-side checks of branch rollouts (mt_rollout_branches, BatchedEnvs.rollout_branches) that need no device.

- mt_rollout_branches' argument errors, which it reports before it looks at the handle.
- BatchedEnvs.rollout_branches' ValueErrors and the shape / dtype checks of `out`, raised before the library is called.
"""
import math

import numpy as np
import pytest

from manytor_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


A16, A4 = 0x10000, 0x10004              # never dereferenced: every case fails before the handle is looked at

#        n_steps, n_branches, src, actions, gamma, return, length, done, obs
GOOD = (4, 8, A16, A16, 0.99, A16, A16, A16, A16)


def _with(**kw):
    names = ("n_steps", "n_branches", "src", "actions", "gamma", "ret", "length", "done", "obs")
    args = dict(zip(names, GOOD))
    args.update(kw)
    return tuple(args[n] for n in names)


@pytest.mark.parametrize("args, message", [
    (_with(n_steps=-1), b"n_steps must be in [0, 4096]"),
    (_with(n_steps=4097), b"n_steps must be in [0, 4096]"),
    (_with(n_steps=-1, src=None, actions=A4), b"n_steps must be in [0, 4096]"),
    (_with(n_branches=-1), b"n_branches must be in [0, 2000000000]"),
    (_with(n_branches=2000000001), b"n_branches must be in [0, 2000000000]"),
    (_with(gamma=math.nan), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=-0.1), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=1.5), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=math.inf), b"gamma must be finite and in [0, 1]"),
    (_with(src=None), b"src_dev is NULL"),
    (_with(src=A4), b"src_dev must be 16-byte aligned"),
    (_with(actions=None), b"actions_dev is NULL"),
    (_with(actions=A4), b"actions_dev must be 16-byte aligned"),
    (_with(ret=None), b"return_dev is NULL"),
    (_with(ret=A4), b"return_dev must be 16-byte aligned"),
    (_with(length=None), b"length_dev is NULL"),
    (_with(length=A4), b"length_dev must be 16-byte aligned"),
    (_with(done=None), b"done_dev is NULL"),
    (_with(done=A4), b"done_dev must be 16-byte aligned"),
    (_with(obs=A4), b"obs_dev must be 16-byte aligned"),
    (_with(obs=None), b"env is NULL"),                      # obs_dev is optional
    (_with(), b"env is NULL"),
    (_with(n_steps=0, n_branches=0, gamma=0.0), b"env is NULL"),
    (_with(n_steps=4096, n_branches=2000000000, gamma=1.0), b"env is NULL"),
])
def test_mt_rollout_branches_argument_errors(lib, args, message):
    assert lib.mt_rollout_branches(None, *args, None) == -1     # MT_ERR_INVALID
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
    env.cfg = _lib.MtConfig()
    return env


def _out(m, obs=True, obs_dtype=None, obs_shape=None, ret_dtype=None, len_dtype=None, done_dtype=None, done_shape=None):
    import torch
    from manytor_b200 import Branches
    return Branches(torch.zeros((m,), dtype=ret_dtype or torch.float32),
                    torch.zeros((m,), dtype=len_dtype or torch.int32),
                    torch.zeros(done_shape or (m,), dtype=done_dtype or torch.uint8),
                    torch.zeros(obs_shape or (m, 30), dtype=obs_dtype or torch.float32) if obs else None)


def test_rollout_branches_checks_run_before_the_library(monkeypatch):
    import torch
    from manytor_b200 import FinalInfo
    env = _envs_without_library(monkeypatch)
    act = np.zeros((3, 5, 4), np.float32)
    src = np.array([0, 1, 1, 7, 2])
    cases = [
        (dict(actions=np.zeros((3, 5), np.float32), src=src), r"actions must have shape \(K, M, 4\)"),
        (dict(actions=np.zeros((3, 5, 3), np.float32), src=src), r"actions must have shape \(K, M, 4\)"),
        (dict(actions=np.zeros((4097, 1, 4), np.float32), src=[0]), "at most 4096 steps"),
        (dict(actions=act), "src=None branches every env once"),
        (dict(actions=act, src=src[:4]), r"src must have shape \(5,\)"),
        (dict(actions=act, src=src.reshape(5, 1)), r"src must have shape \(5,\)"),
        (dict(actions=act, src=src.astype(np.float32)), "src must hold integers"),
        (dict(actions=act, src=torch.zeros(5, dtype=torch.bool)), "src must hold integers"),
        (dict(actions=act, src=src, gamma=math.nan), "gamma must be finite and in"),
        (dict(actions=act, src=src, gamma=-0.1), "gamma must be finite and in"),
        (dict(actions=act, src=src, gamma=1.5), "gamma must be finite and in"),
        (dict(actions=act, src=src, out=(None, None, None, None)), "out must be a Branches"),
        (dict(actions=act, src=src, out=FinalInfo(None, None, None)), "out must be a Branches"),
        (dict(actions=act, src=src, out=_out(5)), r"out.obs must be None here \(write_obs=False\)"),
        (dict(actions=act, src=src, write_obs=True, out=_out(5, obs=False)), "out.obs must be a tensor"),
        (dict(actions=act, src=src, write_obs=True, out=_out(5, obs_dtype=torch.float16)),
         r"out.obs must have shape \(5, 30\) and dtype torch.float32"),
        (dict(actions=act, src=src, write_obs=True, out=_out(5, obs_shape=(5, 29))), "out.obs must have shape"),
        (dict(actions=act, src=src, out=_out(4, obs=False)), r"out.ret must have shape \(5,\)"),
        (dict(actions=act, src=src, out=_out(5, obs=False, ret_dtype=torch.float64)),
         r"out.ret must have shape \(5,\) and dtype torch.float32"),
        (dict(actions=act, src=src, out=_out(5, obs=False, len_dtype=torch.int64)),
         r"out.length must have shape \(5,\) and dtype torch.int32"),
        (dict(actions=act, src=src, out=_out(5, obs=False, done_dtype=torch.bool)),
         r"out.done must have shape \(5,\) and dtype torch.uint8"),
        (dict(actions=act, src=src, out=_out(5, obs=False, done_shape=(5, 1))), "out.done must have shape"),
        (dict(actions=act, src=src, out=_out(5, obs=False)._replace(ret=None)), "out.ret must be a tensor"),
    ]
    for kw, message in cases:
        with pytest.raises(ValueError, match=message):
            env.rollout_branches(**kw)
    env16 = _envs_without_library(monkeypatch, torch.float16)
    with pytest.raises(ValueError, match=r"out.obs must have shape \(5, 30\) and dtype torch.float16"):
        env16.rollout_branches(act, src, write_obs=True, out=_out(5))
    # right shape and dtype, but not contiguous: still refused before the library
    strided = _out(5)._replace(obs=torch.zeros((5, 60))[:, ::2])
    with pytest.raises(ValueError, match="out.obs must be a contiguous tensor on cpu"):
        env.rollout_branches(act, src, write_obs=True, out=strided)
    # nothing to do: no library call, and the buffers come back untouched
    for a, s in ((np.zeros((0, 5, 4), np.float32), src), (np.zeros((3, 0, 4), np.float32), np.zeros(0, np.int64))):
        pre = _out(a.shape[1], obs=False)
        pre.ret.fill_(7.0)
        got = env.rollout_branches(a, s, out=pre)
        assert got is pre and bool((got.ret == 7.0).all())
