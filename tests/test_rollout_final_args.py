"""CPU-side checks of trajectory rollouts with final outputs (mt_rollout_final, BatchedEnvs.rollout(final=True)) that
need no device.

- mt_rollout_final's argument errors, which it reports before it looks at the handle, in mt_rollout's order and then
  mt_step_final's.
- BatchedEnvs.rollout(final=True)'s ValueErrors and the shape / dtype checks of `final_out`, raised before the
  library is called.
"""
import numpy as np
import pytest

from manytor_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


A16, A4 = 0x10000, 0x10004              # never dereferenced: every case fails before the handle is looked at


#  n_steps, actions, drawn, obs, reward, done, final_obs, final_return, final_length
@pytest.mark.parametrize("args, message", [
    ((-1, A16, None, A16, A16, A16, A16, A16, A16), b"n_steps < 0"),
    ((-1, A4, None, None, None, None, None, None, None), b"n_steps < 0"),
    ((4, A4, None, A16, A16, A16, A16, A16, A16), b"actions_dev must be 16-byte aligned"),
    ((4, None, A4, A16, A16, A16, A16, A16, A16), b"drawn_dev must be 16-byte aligned"),
    ((4, A16, A16, A16, A16, A16, A16, A16, A16), b"drawn_dev must be NULL when actions_dev is given"),
    ((4, None, None, None, A16, A16, A16, A16, A16), b"obs_dev is NULL"),
    ((4, None, None, A4, A16, A16, A16, A16, A16), b"obs_dev must be 16-byte aligned"),
    ((4, None, None, A16, None, A16, A16, A16, A16), b"reward_dev is NULL"),
    ((4, None, None, A16, A4, A16, A16, A16, A16), b"reward_dev must be 16-byte aligned"),
    ((4, None, None, A16, A16, None, A16, A16, A16), b"done_dev is NULL"),
    ((4, None, None, A16, A16, A4, A16, A16, A16), b"done_dev must be 16-byte aligned"),
    ((4, None, None, A16, A16, A16, None, A16, A16), b"final_obs_dev is NULL"),
    ((4, None, None, A16, A16, A16, A4, A16, A16), b"final_obs_dev must be 16-byte aligned"),
    ((4, None, None, A16, A16, A16, A16, None, A16), b"final_return_dev is NULL"),
    ((4, None, None, A16, A16, A16, A16, A4, A16), b"final_return_dev must be 16-byte aligned"),
    ((4, None, None, A16, A16, A16, A16, A16, None), b"final_length_dev is NULL"),
    ((4, None, None, A16, A16, A16, A16, A16, A4), b"final_length_dev must be 16-byte aligned"),
    ((4, None, A4, None, None, None, None, None, None), b"drawn_dev must be 16-byte aligned"),
    ((4, A16, None, A16, A16, A16, A16, A16, A16), b"env is NULL"),
    ((0, None, A16, A16, A16, A16, A16, A16, A16), b"env is NULL"),
])
def test_mt_rollout_final_argument_errors(lib, args, message):
    assert lib.mt_rollout_final(None, *args, None) == -1     # MT_ERR_INVALID
    assert message in lib.mt_last_error()


def _envs_without_library(monkeypatch, obs_dtype=None, auto_reset=True):
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
    env.cfg.auto_reset = int(auto_reset)
    return env


def _final(k, obs_dtype=None, obs_shape=None, ret_dtype=None, len_dtype=None, len_shape=None):
    import torch
    from manytor_b200 import FinalInfo
    return FinalInfo(torch.zeros(obs_shape or (k, 8, 30), dtype=obs_dtype or torch.float32),
                     torch.zeros((k, 8), dtype=ret_dtype or torch.float32),
                     torch.zeros(len_shape or (k, 8), dtype=len_dtype or torch.int32))


def test_rollout_final_checks_run_before_the_library(monkeypatch):
    import torch
    from manytor_b200 import Trajectory
    env = _envs_without_library(monkeypatch)
    act = np.zeros((3, 8, 4), np.float32)
    with pytest.raises(ValueError, match="final=True needs write_obs=True"):
        env.rollout(act, write_obs=False, final=True)
    with pytest.raises(ValueError, match="final=True needs a handle created with auto_reset=True"):
        _envs_without_library(monkeypatch, auto_reset=False).rollout(act, final=True)
    with pytest.raises(ValueError, match="final=True needs a handle created with auto_reset=True"):
        _envs_without_library(monkeypatch, auto_reset=False).rollout(n_steps=3, final=True)
    cases = [
        (dict(actions=act, final_out=_final(3)), "final_out needs final=True"),
        (dict(actions=act, final=True, final_out=(None, None, None)), "final_out must be a FinalInfo"),
        (dict(actions=act, final=True, final_out=Trajectory(None, None, None, None)), "final_out must be a FinalInfo"),
        (dict(actions=act, final=True, final_out=_final(3, obs_dtype=torch.float16)),
         r"final_out.obs must have shape \(3, 8, 30\) and dtype torch.float32"),
        (dict(actions=act, final=True, final_out=_final(3, obs_shape=(3, 8, 29))), "final_out.obs must have shape"),
        (dict(actions=act, final=True, final_out=_final(4)), "final_out.obs must have shape"),
        (dict(n_steps=3, final=True, final_out=_final(3, ret_dtype=torch.float64)),
         r"final_out.episode_return must have shape \(3, 8\) and dtype torch.float32"),
        (dict(n_steps=3, final=True, final_out=_final(3, len_dtype=torch.int64)),
         r"final_out.episode_length must have shape \(3, 8\) and dtype torch.int32"),
        (dict(n_steps=3, final=True, final_out=_final(3, len_shape=(3, 9))), "final_out.episode_length must have shape"),
        (dict(n_steps=3, final=True, final_out=_final(3)._replace(episode_return=None)),
         "final_out.episode_return must be a tensor"),
        # the Trajectory's own checks still apply
        (dict(actions=act, final=True, out=(None, None, None, None)), "out must be a Trajectory"),
    ]
    for kw, message in cases:
        with pytest.raises(ValueError, match=message):
            env.rollout(**kw)
    env16 = _envs_without_library(monkeypatch, torch.float16)
    with pytest.raises(ValueError, match=r"final_out.obs must have shape \(3, 8, 30\) and dtype torch.float16"):
        env16.rollout(act, final=True, final_out=_final(3))
    # right shape and dtype, but not contiguous: still refused before the library
    strided = _final(3)._replace(obs=torch.zeros((3, 8, 60))[:, :, ::2])
    with pytest.raises(ValueError, match="final_out.obs must be a contiguous tensor on cpu"):
        env.rollout(act, final=True, final_out=strided)
