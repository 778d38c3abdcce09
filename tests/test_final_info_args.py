"""CPU-side checks of the final outputs of a step (mt_step_final, BatchedEnvs.step(final=True),
ManyTorVectorEnv(final_info=True)) that need no device.

- mt_step_final's argument errors, which it reports before it looks at the handle.
- BatchedEnvs.step(final=True)'s ValueErrors, raised before the library is called.
- The Gymnasium adapter's final_info flag: which step it asks for and the info it builds.
"""
import pytest

from manytor_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


A16, A4 = 0x10000, 0x10004              # never dereferenced: every case fails before the handle is looked at


@pytest.mark.parametrize("args, message", [
    ((None, A16, A16, A16, None, A16, A16, A16), b"actions_dev is NULL"),
    ((A4, A16, A16, A16, None, A16, A16, A16), b"actions_dev must be 16-byte aligned"),
    ((A16, None, A16, A16, None, A16, A16, A16), b"obs_dev is NULL"),
    ((A16, A4, A16, A16, None, A16, A16, A16), b"obs_dev must be 16-byte aligned"),
    ((A16, A16, None, A16, None, A16, A16, A16), b"reward_dev/done_dev is NULL"),
    ((A16, A16, A16, None, None, A16, A16, A16), b"reward_dev/done_dev is NULL"),
    ((A16, A16, A16, A16, None, None, A16, A16), b"final_obs_dev is NULL"),
    ((A16, A16, A16, A16, None, A4, A16, A16), b"final_obs_dev must be 16-byte aligned"),
    ((A16, A16, A16, A16, None, A16, None, A16), b"final_return_dev is NULL"),
    ((A16, A16, A16, A16, None, A16, A4, A16), b"final_return_dev must be 16-byte aligned"),
    ((A16, A16, A16, A16, None, A16, A16, None), b"final_length_dev is NULL"),
    ((A16, A16, A16, A16, None, A16, A16, A4), b"final_length_dev must be 16-byte aligned"),
    ((A16, A16, A16, A16, A16, A16, A16, A16), b"env is NULL"),
])
def test_mt_step_final_argument_errors(lib, args, message):
    assert lib.mt_step_final(None, *args, None) == -1     # MT_ERR_INVALID
    assert message in lib.mt_last_error()


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name})")


def _envs_without_library(monkeypatch, auto_reset=True):
    """A BatchedEnvs of 8 envs, X = 10, J = 4 whose library calls fail the test."""
    import torch
    from manytor_b200 import core

    def no_load(*a, **k):
        raise AssertionError("the library was loaded")

    monkeypatch.setattr(core._lib, "load", no_load)
    env = object.__new__(core.BatchedEnvs)
    env._h = None
    env._lib = _NoLibrary()
    env.n, env.x, env.j = 8, 10, 4
    env.obs_dtype = torch.float32
    env.device = torch.device("cpu")
    env.cfg = _lib.MtConfig()
    env.cfg.auto_reset = int(auto_reset)
    return env


def test_step_final_checks_run_before_the_library(monkeypatch):
    import numpy as np
    act = np.zeros((8, 4), np.float32)
    env = _envs_without_library(monkeypatch)
    with pytest.raises(ValueError, match="final=True needs write_obs=True"):
        env.step(act, write_obs=False, final=True)
    with pytest.raises(ValueError, match="final=True needs a handle created with auto_reset=True"):
        _envs_without_library(monkeypatch, auto_reset=False).step(act, final=True)


def test_final_info_is_exported():
    import manytor_b200
    assert manytor_b200.FinalInfo._fields == ("obs", "episode_return", "episode_length")
    assert "FinalInfo" in manytor_b200.__all__


class _RecordingEnvs:
    """Stands in for BatchedEnvs: records how step was called and returns CPU tensors."""

    def __init__(self, n=4, x=2):
        self.n, self.x, self.calls = n, x, []

    def step(self, actions, **kw):
        import torch
        from manytor_b200 import FinalInfo
        self.calls.append(kw)
        obs = torch.zeros((self.n, 3 * self.x))
        rew = torch.zeros(self.n)
        done = torch.tensor([0, 1, 2, 0], dtype=torch.uint8)
        if kw.get("final"):
            return obs, rew, done, FinalInfo(torch.ones((self.n, 3 * self.x)), torch.full((self.n,), 3.0),
                                             torch.full((self.n,), 7, dtype=torch.int32))
        return obs, rew, done


def _adapter(final_info):
    from manytor_b200 import ManyTorVectorEnv
    venv = object.__new__(ManyTorVectorEnv)
    venv.final_info = final_info
    venv.envs = _RecordingEnvs()
    return venv


def test_vector_env_final_info_flag():
    import inspect
    import torch
    from manytor_b200 import ManyTorVectorEnv
    assert inspect.signature(ManyTorVectorEnv).parameters["final_info"].default is False
    venv = _adapter(False)
    *_, info = venv.step(None)
    assert info == {} and venv.envs.calls == [{}]          # the default: plain mt_step, empty info
    venv = _adapter(True)
    obs, rew, term, trunc, info = venv.step(None)
    assert venv.envs.calls == [{"final": True}]
    mask = torch.tensor([False, True, True, False])
    assert torch.equal(term, torch.tensor([False, True, False, False]))
    assert torch.equal(trunc, torch.tensor([False, False, True, False]))
    assert set(info) == {"final_obs", "_final_obs", "episode", "_episode"}
    assert torch.equal(info["_final_obs"], mask) and torch.equal(info["_episode"], mask)
    assert info["final_obs"].shape == (4, 6)
    assert torch.equal(info["episode"]["r"], torch.full((4,), 3.0))
    assert info["episode"]["l"].dtype == torch.int32
