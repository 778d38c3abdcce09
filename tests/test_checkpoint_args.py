"""CPU-side checks of the reset-count exchange (mt_get/set_reset_counts, BatchedEnvs.get/set_state's `resets`) that
need no device: argument errors, which are reported before the handle is looked at, and the shape check of
set_state(resets=...), which runs before the library is called."""
import numpy as np
import pytest

from manytor_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    build.build()                       # no-op when up to date
    return _lib.load()


A16 = 0x10000                           # never dereferenced: every case fails before the handle is looked at


@pytest.mark.parametrize("env, counts, message", [
    (None, None, b"counts_dev is NULL"),
    (A16, None, b"counts_dev is NULL"),
    (None, A16, b"env is NULL"),
])
def test_reset_count_argument_errors(lib, env, counts, message):
    assert lib.mt_get_reset_counts(env, counts, None) == -1           # MT_ERR_INVALID
    assert message in lib.mt_last_error()
    assert lib.mt_set_reset_counts(env, counts, None, None) == -1
    assert message in lib.mt_last_error()


def test_set_state_checks_resets_before_the_library(monkeypatch):
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
    env.device = torch.device("cpu")
    for bad in (np.zeros(7, np.int64), np.zeros((8, 1), np.int32), torch.zeros(9, dtype=torch.int32), [1, 2, 3],
                np.int64(5)):
        with pytest.raises(ValueError, match=r"resets must have shape \(8,\)"):
            env.set_state(resets=bad)
        with pytest.raises(ValueError, match=r"resets must have shape \(8,\)"):
            env.set_state(goals=np.zeros((8, 4), np.float32), resets=bad, mask=np.ones(8, bool))
