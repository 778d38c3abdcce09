"""CPU-side checks of in-kernel branch draws (mt_rollout_branches_random, mt_branch_actions and their BatchedEnvs
methods) that need no device.

- The argument errors of both entry points, which they report before they look at the handle.
- BatchedEnvs.rollout_branches(n_steps=..., draw_key=...) and BatchedEnvs.branch_actions' ValueErrors, raised before the
  library is called.
"""
import math

import numpy as np
import pytest

from manytor_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


A16, A8, A4 = 0x10000, 0x10008, 0x10004  # never dereferenced: every case fails before the handle is looked at

#        n_steps, n_prefix, n_branches, src, prefix, key, gamma, return, length, done, obs
GOOD = (4, 2, 8, A16, A16, A16, 0.99, A16, A16, A16, A16)
NAMES = ("n_steps", "n_prefix", "n_branches", "src", "prefix", "key", "gamma", "ret", "length", "done", "obs")


def _with(**kw):
    args = dict(zip(NAMES, GOOD))
    args.update(kw)
    return tuple(args[n] for n in NAMES)


@pytest.mark.parametrize("args, message", [
    (_with(n_steps=-1), b"n_steps must be in [0, 4096]"),
    (_with(n_steps=4097), b"n_steps must be in [0, 4096]"),
    (_with(n_steps=4097, n_prefix=4097), b"n_steps must be in [0, 4096]"),
    (_with(n_steps=-1, src=None, key=None), b"n_steps must be in [0, 4096]"),
    (_with(n_prefix=-1), b"n_prefix must be in [0, n_steps]"),
    (_with(n_prefix=5), b"n_prefix must be in [0, n_steps]"),
    (_with(n_steps=0, n_prefix=1), b"n_prefix must be in [0, n_steps]"),
    (_with(n_prefix=5, n_branches=-1), b"n_prefix must be in [0, n_steps]"),
    (_with(n_branches=-1), b"n_branches must be in [0, 2000000000]"),
    (_with(n_branches=2000000001), b"n_branches must be in [0, 2000000000]"),
    (_with(gamma=math.nan), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=-0.1), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=1.5), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=math.inf), b"gamma must be finite and in [0, 1]"),
    (_with(gamma=math.nan, src=None), b"gamma must be finite and in [0, 1]"),
    (_with(src=None), b"src_dev is NULL"),
    (_with(src=A4), b"src_dev must be 16-byte aligned"),
    (_with(src=A8), b"src_dev must be 16-byte aligned"),
    (_with(prefix=None), b"prefix_dev is NULL"),
    (_with(prefix=A4), b"prefix_dev must be 16-byte aligned"),
    (_with(n_prefix=0), b"prefix_dev must be NULL when n_prefix is 0"),
    (_with(n_prefix=0, prefix=A4), b"prefix_dev must be 16-byte aligned"),
    (_with(key=None), b"draw_key_dev is NULL"),
    (_with(key=A4), b"draw_key_dev must be 8-byte aligned"),
    (_with(key=A4 + 1), b"draw_key_dev must be 8-byte aligned"),
    (_with(prefix=None, key=None), b"prefix_dev is NULL"),
    (_with(key=None, ret=None), b"draw_key_dev is NULL"),
    (_with(ret=None), b"return_dev is NULL"),
    (_with(ret=A4), b"return_dev must be 16-byte aligned"),
    (_with(length=None), b"length_dev is NULL"),
    (_with(length=A4), b"length_dev must be 16-byte aligned"),
    (_with(done=None), b"done_dev is NULL"),
    (_with(done=A4), b"done_dev must be 16-byte aligned"),
    (_with(obs=A4), b"obs_dev must be 16-byte aligned"),
    (_with(obs=None), b"env is NULL"),                      # obs_dev is optional
    (_with(key=A8), b"env is NULL"),                        # the key needs 8-byte alignment only
    (_with(n_prefix=0, prefix=None), b"env is NULL"),
    (_with(n_prefix=4), b"env is NULL"),                    # a prefix of every step
    (_with(), b"env is NULL"),
    (_with(n_steps=0, n_prefix=0, prefix=None, n_branches=0, gamma=0.0), b"env is NULL"),
    (_with(n_steps=4096, n_prefix=4096, n_branches=2000000000, gamma=1.0), b"env is NULL"),
])
def test_mt_rollout_branches_random_argument_errors(lib, args, message):
    assert lib.mt_rollout_branches_random(None, *args, None) == -1     # MT_ERR_INVALID
    assert message in lib.mt_last_error()


#        key, first_step, n_steps, n_rows, branches, out
GOOD_BA = (A16, 0, 3, 8, A16, A16)


def _ba(**kw):
    args = dict(zip(("key", "first", "n_steps", "rows", "ids", "out"), GOOD_BA))
    args.update(kw)
    return args["key"], args["first"], args["n_steps"], args["rows"], args["ids"], args["out"]


@pytest.mark.parametrize("args, message", [
    (_ba(key=None), b"draw_key_dev is NULL"),
    (_ba(key=A4), b"draw_key_dev must be 8-byte aligned"),
    (_ba(key=None, first=-1), b"draw_key_dev is NULL"),
    (_ba(first=-1), b"first_step must be >= 0"),
    (_ba(first=-(2 ** 31)), b"first_step must be >= 0"),
    (_ba(first=-1, n_steps=-1), b"first_step must be >= 0"),
    (_ba(n_steps=-1), b"n_steps must be >= 0"),
    (_ba(rows=-1), b"n_rows must be in [0, 2000000000]"),
    (_ba(rows=2000000001), b"n_rows must be in [0, 2000000000]"),
    (_ba(ids=None), b"branch_dev is NULL"),
    (_ba(ids=A8), b"branch_dev must be 16-byte aligned"),
    (_ba(out=None), b"out_dev is NULL"),
    (_ba(out=A4), b"out_dev must be 16-byte aligned"),
    (_ba(key=A8), b"env is NULL"),
    (_ba(), b"env is NULL"),
    (_ba(first=2 ** 31 - 1, n_steps=2 ** 31 - 1, rows=2000000000), b"env is NULL"),
    (_ba(n_steps=0, rows=0), b"env is NULL"),
])
def test_mt_branch_actions_argument_errors(lib, args, message):
    assert lib.mt_branch_actions(None, *args, None) == -1      # MT_ERR_INVALID
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


def _out(m, obs=False):
    import torch
    from manytor_b200 import Branches
    return Branches(torch.zeros((m,), dtype=torch.float32), torch.zeros((m,), dtype=torch.int32),
                    torch.zeros((m,), dtype=torch.uint8), torch.zeros((m, 30)) if obs else None)


def test_rollout_branches_draw_checks_run_before_the_library(monkeypatch):
    import torch
    env = _envs_without_library(monkeypatch)
    src = np.array([0, 1, 1, 7, 2])
    pre = np.zeros((2, 5, 4), np.float32)
    cases = [
        (dict(actions=None, src=src, n_steps=4), "need an explicit draw_key"),
        (dict(actions=pre, src=src, n_steps=4), "need an explicit draw_key"),
        (dict(actions=None, src=src, n_steps=4, draw_key=1.0), "draw_key must be an int or a"),
        (dict(actions=None, src=src, n_steps=4, draw_key=True), "draw_key must be an int or a"),
        (dict(actions=None, src=src, n_steps=4, draw_key="7"), "draw_key must be an int or a"),
        (dict(actions=None, src=src, n_steps=4, draw_key=torch.zeros(1, dtype=torch.int32)),
         r"draw_key must be an int or a \(1,\) int64 tensor"),
        (dict(actions=None, src=src, n_steps=4, draw_key=torch.zeros(2, dtype=torch.int64)),
         r"draw_key must be an int or a \(1,\) int64 tensor"),
        (dict(actions=None, src=src, n_steps=4, draw_key=torch.zeros((), dtype=torch.int64)),
         r"draw_key must be an int or a \(1,\) int64 tensor"),
        (dict(actions=None, src=src, n_steps=4097, draw_key=0), r"n_steps must be in \[0, 4096\]"),
        (dict(actions=None, src=src, draw_key=0), "n_steps is required when actions is None"),
        (dict(actions=None, draw_key=torch.zeros(1, dtype=torch.int64)), "n_steps is required when actions is None"),
        (dict(actions=None, src=src, n_steps=-1, draw_key=0), r"n_steps must be in \[0, 4096\]"),
        (dict(actions=pre, src=src, n_steps=1, draw_key=0), "the prefix has 2 steps, more than n_steps = 1"),
        (dict(actions=np.zeros((2, 5, 3), np.float32), src=src, n_steps=4, draw_key=0),
         r"a prefix of actions must have shape \(P, 5, 4\)"),
        (dict(actions=np.zeros((2, 4, 4), np.float32), src=src, n_steps=4, draw_key=0),
         r"a prefix of actions must have shape \(P, 5, 4\)"),
        (dict(actions=np.zeros((5, 4), np.float32), src=src, n_steps=4, draw_key=0), "a prefix of actions must have"),
        (dict(actions=np.zeros((2, 5, 4), np.float32), n_steps=4, draw_key=0),
         r"a prefix of actions must have shape \(P, 8, 4\) \(M = N\)"),
        (dict(actions=None, src=src.reshape(5, 1), n_steps=4, draw_key=0), r"src must have shape \(M,\)"),
        (dict(actions=None, src=src.astype(np.float32), n_steps=4, draw_key=0), "src must hold integers"),
        (dict(actions=None, src=torch.zeros(5, dtype=torch.bool), n_steps=4, draw_key=0), "src must hold integers"),
        (dict(actions=None, src=src, n_steps=4, draw_key=0, gamma=math.nan), "gamma must be finite and in"),
        (dict(actions=None, src=src, n_steps=4, draw_key=0, gamma=1.5), "gamma must be finite and in"),
        (dict(actions=None, src=src, n_steps=4, draw_key=0, out=_out(4)), r"out.ret must have shape \(5,\)"),
        (dict(actions=None, src=src, n_steps=4, draw_key=0, out=_out(5, obs=True)), "out.obs must be None here"),
        (dict(actions=None, src=src, n_steps=4, draw_key=0, write_obs=True, out=_out(5)), "out.obs must be a tensor"),
        (dict(actions=None, n_steps=4, draw_key=0, out=_out(5)), r"out.ret must have shape \(8,\)"),
    ]
    for kw, message in cases:
        with pytest.raises(ValueError, match=message):
            env.rollout_branches(**kw)
    # nothing to do (K = 0 or M = 0): no library call, buffers untouched
    for kw in (dict(actions=None, src=src, n_steps=0, draw_key=5),
               dict(actions=None, src=np.zeros(0, np.int64), n_steps=9, draw_key=2 ** 64 + 5),
               dict(actions=np.zeros((0, 5, 4), np.float32), src=src, n_steps=0, draw_key=-1)):
        pre_out = _out(len(kw["src"]))
        pre_out.ret.fill_(7.0)
        got = env.rollout_branches(out=pre_out, **kw)
        assert got is pre_out and bool((got.ret == 7.0).all())


def test_branch_actions_checks_run_before_the_library(monkeypatch):
    import torch
    env = _envs_without_library(monkeypatch)
    ids = np.array([0, 31, 2 ** 40])
    cases = [
        (dict(branches=ids.reshape(3, 1), draw_key=0, n_steps=2), r"branches must have shape \(M,\)"),
        (dict(branches=5, draw_key=0, n_steps=2), r"branches must have shape \(M,\)"),
        (dict(branches=ids.astype(np.float64), draw_key=0, n_steps=2), "branches must hold integers"),
        (dict(branches=ids, draw_key=None, n_steps=2), "draw_key must be an int or a"),
        (dict(branches=ids, draw_key=0.0, n_steps=2), "draw_key must be an int or a"),
        (dict(branches=ids, draw_key=torch.zeros(1, dtype=torch.uint8), n_steps=2), "draw_key must be an int or a"),
        (dict(branches=ids, draw_key=0, n_steps=-1), r"n_steps must be in \[0, 2\^31\)"),
        (dict(branches=ids, draw_key=0, n_steps=2 ** 31), r"n_steps must be in \[0, 2\^31\)"),
        (dict(branches=ids, draw_key=0, n_steps=1, first_step=-1), r"first_step must be in \[0, 2\^31\)"),
        (dict(branches=ids, draw_key=0, n_steps=1, first_step=2 ** 31), r"first_step must be in \[0, 2\^31\)"),
        (dict(branches=ids, draw_key=0, n_steps=2, out=torch.zeros((2, 3, 3))),
         r"out must be a tensor of shape \(2, 3, 4\) and dtype torch.float32"),
        (dict(branches=ids, draw_key=0, n_steps=2, out=torch.zeros((2, 3, 4), dtype=torch.float64)),
         r"out must be a tensor of shape \(2, 3, 4\)"),
        (dict(branches=ids, draw_key=0, n_steps=2, out=np.zeros((2, 3, 4), np.float32)), "out must be a tensor"),
        (dict(branches=ids, draw_key=0, n_steps=2, out=torch.zeros((2, 3, 8))[:, :, ::2]),
         "out must be a contiguous, 16-byte aligned tensor on cpu"),
    ]
    for kw, message in cases:
        with pytest.raises(ValueError, match=message):
            env.branch_actions(**kw)
    for kw in (dict(branches=ids, draw_key=3, n_steps=0), dict(branches=np.zeros(0, np.int64), draw_key=3, n_steps=4)):
        got = env.branch_actions(**kw)
        assert tuple(got.shape) == (kw["n_steps"], len(kw["branches"]), 4)
