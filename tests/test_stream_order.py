"""CPU-side checks of how BatchedEnvs orders its synchronous calls after work on a non-default stream.

The synchronous calls run on the legacy default stream, which does not wait for PyTorch's (non-blocking) streams.
So BatchedEnvs remembers the non-default stream of a handle's last asynchronous call and waits for it before
stats / step_index / fetch_env; on the default stream, and during CUDA-graph capture, it records and waits for
nothing.  Streams and the library are stand-ins here; tests/test_gpu_streams.py runs the real thing on the GPU."""
import ctypes as C

import pytest
import torch


class FakeStream:
    def __init__(self, ptr, log):
        self.cuda_stream, self._log = ptr, log

    def synchronize(self):
        self._log.append(f"wait {self.cuda_stream:#x}")


class RecordingLibrary:
    def __init__(self, log):
        self._log = log

    def __getattr__(self, name):
        if not name.startswith("mt_"):
            raise AttributeError(name)
        return lambda *args: self._log.append(name) or 0


@pytest.fixture
def world(monkeypatch):
    """(env, log, use(stream ptr), capturing flag): a handle with no device behind it."""
    from manytor_b200 import BatchedEnvs
    log, cur, capturing = [], [FakeStream(0, [])], [False]
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: cur[0])
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: capturing[0])
    env = object.__new__(BatchedEnvs)
    env._lib, env._h, env.device = RecordingLibrary(log), C.c_void_p(), torch.device("cuda", 0)
    env.n, env.x, env.j = 8, 3, 4

    def use(ptr):
        cur[0] = FakeStream(ptr, log)
    return env, log, use, capturing


SYNC_CALLS = {
    "stats": (lambda env: env.stats(), "mt_stats_host"),
    "step_index get": (lambda env: env.step_index, "mt_get_step_index"),
    "step_index set": (lambda env: setattr(env, "step_index", 7), "mt_set_step_index"),
    "fetch_env": (lambda env: env.fetch_env(1), "mt_fetch_env"),
}


@pytest.mark.parametrize("call", sorted(SYNC_CALLS))
def test_waits_once_for_the_side_stream_of_the_last_call(world, call):
    env, log, use, _ = world
    fn, name = SYNC_CALLS[call]
    use(0xA1)
    env.clear_stats()                                  # an asynchronous call on a side stream
    use(0)                                             # the caller leaves `with torch.cuda.stream(side)`
    fn(env)
    fn(env)
    assert log == ["mt_stats_clear", "wait 0xa1", name, name]


@pytest.mark.parametrize("call", sorted(SYNC_CALLS))
def test_default_stream_adds_no_wait(world, call):
    env, log, use, _ = world
    fn, name = SYNC_CALLS[call]
    env.clear_stats()
    fn(env)
    use(0xA1)
    env.clear_stats()
    use(0)
    env.clear_stats()                                  # a later call on the default stream is ordered after it
    fn(env)
    assert log == ["mt_stats_clear", name, "mt_stats_clear", "mt_stats_clear", name]


def test_waits_for_the_latest_side_stream(world):
    env, log, use, _ = world
    use(0xA1)
    env.clear_stats()
    use(0xB2)
    env.clear_stats()
    env.stats()
    assert log == ["mt_stats_clear", "mt_stats_clear", "wait 0xb2", "mt_stats_host"]


def test_graph_capture_records_and_waits_for_nothing(world):
    env, log, use, capturing = world
    use(0xC3)
    capturing[0] = True
    env.clear_stats()                                  # captured, not enqueued
    capturing[0] = False
    use(0)
    env.stats()
    assert log == ["mt_stats_clear", "mt_stats_host"]
