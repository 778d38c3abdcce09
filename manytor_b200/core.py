"""Device-level API: N lock-step ManyTor environments resident on one B200.

`BatchedEnvs` owns one C-ABI handle (include/manytor_b200.h) and exposes the
reference's operations (reset / step / action_sample / get_observations,
manytor.py:141-260) on torch CUDA tensors.  torch is plumbing only: device
memory, streams and (in distributed.py) the NCCL process group.  All compute
runs in libmanytor_b200.so; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
import math
import weakref
from collections import namedtuple
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import MantorLibraryError, MtConfig, MtStats, STATS_FIELDS


@dataclass(frozen=True)
class ArmSpec:
    """A DH arm: rows (a, alpha, d, theta_offset) in radians plus the frame
    selectors the reference hard-codes (manytor.py:42-48, 143, 162, 191)."""

    dh: tuple
    obs_frame: int
    ground_frames: tuple
    catch_frame: int
    radius: float = 51.3
    catch_tol: float = 8.0

    @property
    def n_joints(self) -> int:
        return len(self.dh)


REFERENCE_ARM = ArmSpec(
    dh=((0.0, -math.pi / 2, 4.3, 0.0), (0.0, math.pi / 2, 0.0, 0.0),
        (0.0, -math.pi / 2, 24.3, 0.0), (27.0, math.pi / 2, 0.0, -math.pi / 2)),
    obs_frame=3, ground_frames=(3, 4), catch_frame=4)

# BASELINE.json config 5 (UR5-style 6-DOF chain, metres); selectors per SURVEY.md 8(a-FK)
UR5_ARM = ArmSpec(
    dh=((0.0, math.pi / 2, 0.089159, 0.0), (-0.425, 0.0, 0.0, 0.0), (-0.39225, 0.0, 0.0, 0.0),
        (0.0, math.pi / 2, 0.10915, 0.0), (0.0, -math.pi / 2, 0.09465, 0.0), (0.0, 0.0, 0.0823, 0.0)),
    obs_frame=5, ground_frames=(5, 6), catch_frame=6,
    radius=0.81725, catch_tol=0.81725 * 8.0 / 51.3)


# What BatchedEnvs.rollout returns: obs (K, N, 3X) of the handle's obs_dtype or None, reward (K, N) float32,
# done (K, N) uint8, actions (K, N, J) float32 (the caller's, or the recorded draws) or None.
Trajectory = namedtuple("Trajectory", "obs reward done actions")

# What BatchedEnvs.step(final=True) appends: for each env that ended in the step (done != 0), the observation that
# closed its episode (obs2, before the in-kernel reset; (N, 3X) of the handle's obs_dtype), the episode's return
# ((N,) float32) and length ((N,) int32).  Rows of envs that did not end keep what an earlier step left there.
# BatchedEnvs.rollout(final=True) returns one slice per step: (K, N, 3X), (K, N) and (K, N).
FinalInfo = namedtuple("FinalInfo", "obs episode_return episode_length")

# What BatchedEnvs.rollout_branches returns, one row per branch: the discounted return ((M,) float32), the steps executed
# ((M,) int32), the done byte of the ending step ((M,) uint8, 0 if the branch ran every step) and obs2 of the last
# executed step ((M, 3X) of the handle's obs_dtype, or None without write_obs).
Branches = namedtuple("Branches", "ret length done obs")


# observation dtype -> mt_config.obs_dtype
OBS_DTYPES = {torch.float32: _lib.MT_OBS_F32, torch.float16: _lib.MT_OBS_F16}


def obs_format(dtype) -> int:
    """mt_config.obs_dtype of a torch dtype; anything but float32 / float16 (bf16 included) is refused."""
    if dtype not in OBS_DTYPES:
        raise ValueError(f"obs_dtype must be torch.float32 or torch.float16, not {dtype}")
    return OBS_DTYPES[dtype]


def make_config(n_envs: int, obj_number: int, arm: ArmSpec, device: int, env_id_base: int = 0,
                horizon: int = 0, auto_reset: bool = False, terminate_on_ground: bool = False,
                obs_after_reset: bool = False, seed: int = 0, fk_mode: int = 0, substeps: int = 25,
                action_low: int = -180, action_high: int = 180, obs_dtype=torch.float32) -> MtConfig:
    cfg = _lib.default_config()
    cfg.device = int(device)
    cfg.n_envs = int(n_envs)
    cfg.env_id_base = int(env_id_base)
    cfg.n_joints = arm.n_joints
    cfg.n_obj = int(obj_number)
    for i, row in enumerate(arm.dh):
        for k in range(4):
            cfg.dh[i][k] = float(row[k])
    cfg.obs_frame = arm.obs_frame
    cfg.ground_frame_a, cfg.ground_frame_b = arm.ground_frames
    cfg.catch_frame = arm.catch_frame
    cfg.radius = arm.radius
    cfg.catch_tol = arm.catch_tol
    cfg.substeps = int(substeps)
    cfg.horizon = int(horizon)
    cfg.terminate_on_ground = int(bool(terminate_on_ground))
    cfg.auto_reset = int(bool(auto_reset))
    cfg.obs_after_reset = int(bool(obs_after_reset))
    cfg.fk_mode = int(fk_mode)
    cfg.action_low = int(action_low)
    cfg.action_high = int(action_high)
    cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    cfg.obs_dtype = obs_format(obs_dtype)
    return cfg


def _device_index(device) -> int:
    if device is None:
        if not torch.cuda.is_available():
            raise MantorLibraryError("no CUDA device: manytor_b200 needs a B200 (there is no CPU fallback)")
        return torch.cuda.current_device()
    if isinstance(device, int):
        return device
    d = torch.device(device)
    if d.type != "cuda":
        raise MantorLibraryError(f"device {d} is not a CUDA device (there is no CPU fallback)")
    return d.index if d.index is not None else torch.cuda.current_device()


class _PinnedBlock:
    """Owner of one page-locked allocation (mt_host_alloc).  The numpy views handed to callers keep
    it alive through their base chain (view -> ctypes buffer -> block), so the memory is released
    only when the last view is gone -- not when the BatchedEnvs that allocated it is collected."""

    def __init__(self, nbytes: int, alloc=None, free=None):
        if (alloc is None) != (free is None):
            raise ValueError("pass both `alloc` and `free` (tests) or neither (mt_host_alloc / mt_host_free)")
        ptr = C.c_void_p()
        if alloc is None:
            lib = _lib.load()
            self._free = lib.mt_host_free
            _lib.check(lib.mt_host_alloc(C.byref(ptr), max(int(nbytes), 1)))
        else:
            self._free = free
            ptr = C.c_void_p(alloc(max(int(nbytes), 1)))
        self.ptr = ptr.value
        self._finalizer = weakref.finalize(self, self._free, C.c_void_p(self.ptr))


class PinnedArray:
    """A numpy array over page-locked host memory (mt_host_alloc)."""

    def __init__(self, shape, dtype, alloc=None, free=None):
        self.shape = tuple(int(s) for s in shape)
        self.dtype = np.dtype(dtype)
        count = int(np.prod(self.shape))
        nbytes = count * self.dtype.itemsize
        self.block = _PinnedBlock(nbytes, alloc, free)
        buf = (C.c_char * max(nbytes, 1)).from_address(self.block.ptr)
        buf._mt_block = self.block                     # the buffer object is the base of every view below
        self.array = np.frombuffer(buf, dtype=self.dtype, count=count).reshape(self.shape)

    @property
    def ptr(self) -> int:
        return self.block.ptr


class BatchedEnvs:
    """N environments in HBM advanced by one fused kernel per step.

    obs_dtype: torch.float32 (default) or torch.float16.  Every observation this object returns
    (step, observe, reset(returnable=True), rollout_random, step_host) is of that dtype; float16
    observations are the float32 ones rounded to nearest even, written by the kernels themselves
    (half the bytes to HBM and across PCIe)."""

    _side = None                                           # non-default stream of the last enqueued call (_stream)

    def __init__(self, n_envs: int, obj_number: int = 10, arm: ArmSpec = REFERENCE_ARM, device=None,
                 env_id_base: int = 0, horizon: int = 0, auto_reset: bool = False,
                 terminate_on_ground: bool = False, obs_after_reset: bool = False, seed: int = 0,
                 fk_mode: int = 0, substeps: int = 25, action_low: int = -180, action_high: int = 180,
                 lib_path: Optional[str] = None, obs_dtype=torch.float32):
        obs_format(obs_dtype)
        self.obs_dtype = obs_dtype
        self._lib = _lib.load(lib_path)
        self._h = C.c_void_p()
        dev = _device_index(device)
        self.device = torch.device("cuda", dev)
        self.arm = arm
        self.n, self.x, self.j = int(n_envs), int(obj_number), arm.n_joints
        self.cfg = make_config(n_envs, obj_number, arm, dev, env_id_base, horizon, auto_reset,
                               terminate_on_ground, obs_after_reset, seed, fk_mode, substeps,
                               action_low, action_high, obs_dtype)
        _lib.check(self._lib.mt_create(C.byref(self.cfg), C.byref(self._h)))
        self._obs = self._reward = self._done = self._joints = self._actions = self._final = None
        self._stream_keepalive = None
        self._pinned = {}
        self._pinned_ptr = {}                              # id(array) -> address, for the arrays in _pinned (kept alive there)
        self._host_io = {}                                 # write_obs -> step_host's buffers and their addresses

    # -- plumbing -------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.mt_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        """The current stream, for an asynchronous call.  A non-default stream is remembered (not while a CUDA
        graph is being captured: a capture enqueues nothing) so that the synchronous calls can wait for it."""
        s = torch.cuda.current_stream(self.device)
        if not s.cuda_stream:
            self._side = None
        elif not torch.cuda.is_current_stream_capturing():
            self._side = s
        return C.c_void_p(s.cuda_stream)

    def _after_side_stream(self):
        """Before a call that runs on the legacy default stream or on the handle's own streams (stats, step_index,
        fetch_env, step_host): wait for this handle's work on a non-default stream.  The legacy stream does not
        wait for PyTorch's streams (they are non-blocking), so without this such a call could run before the work
        it is meant to see.  Work on the default stream is already ordered: nothing to do there."""
        if self._side is not None and not torch.cuda.is_current_stream_capturing():
            self._side.synchronize()
            self._side = None

    def _empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def _as_dev(self, a, dtype, shape=None):
        t = torch.as_tensor(a)
        t = t.to(device=self.device, dtype=dtype).contiguous()
        if shape is not None:
            t = t.reshape(shape)
        return t

    @staticmethod
    def _p(t: Optional[torch.Tensor]):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    def _mask(self, mask):
        if mask is None:
            return None
        return self._as_dev(mask, torch.bool, (self.n,)).view(torch.uint8)

    def _out_buffers(self, want_obs=True, want_joints=False, want_final=False):
        if self._reward is None:
            self._reward = self._empty((self.n,), torch.float32)
            self._done = self._empty((self.n,), torch.uint8)
        if want_obs and self._obs is None:
            self._obs = self._empty((self.n, 3 * self.x), self.obs_dtype)
        if want_joints and self._joints is None:
            self._joints = self._empty((self.n, self.j, 3), torch.float32)
        if want_final and self._final is None:
            self._final = FinalInfo(self._empty((self.n, 3 * self.x), self.obs_dtype),
                                    self._empty((self.n,), torch.float32), self._empty((self.n,), torch.int32))

    # -- reference operations --------------------------------------------------
    def reset(self, mask=None, returnable: bool = False):
        """Environment.reset / Multienv.reset (manytor.py:219-253, 106-109)."""
        m = self._mask(mask)
        _lib.check(self._lib.mt_reset(self._h, self._p(m), self._stream()))
        if returnable:
            # the same storage `step` writes its observations to: a policy that holds on to the tensor
            # returned here keeps seeing fresh observations (examples/policy_loop.py)
            self._out_buffers()
            return self.observe(out=self._obs)
        return None

    def observe(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Environment.get_observations (manytor.py:141-153) for every env -> (N, 3X) of obs_dtype."""
        if out is None:
            out = self._empty((self.n, 3 * self.x), self.obs_dtype)
        elif out.dtype != self.obs_dtype:
            raise ValueError(f"observe(out=...) needs a {self.obs_dtype} buffer (this handle's obs_dtype), got {out.dtype}")
        _lib.check(self._lib.mt_observe(self._h, self._p(out), self._stream()))
        return out

    def step(self, actions, joints: bool = False, write_obs: bool = True, final: bool = False):
        """Environment.step / Multienv.step (manytor.py:255-260, 115-122).

        actions: (N, J) degrees.  Returns (obs (N,3X) obs_dtype, reward (N,) f32,
        done (N,) u8 [, joints (N,J,3)] [, FinalInfo]) -- views of buffers this object
        reuses on the next step.

        final=True (mt_step_final; needs auto_reset and write_obs) appends a FinalInfo: the
        last observation, return and length of every episode that ended in this step, in the
        rows where done != 0, which the in-kernel reset would otherwise discard.
        """
        if final:
            self._check_final(write_obs)
        if (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.float32
                and actions.is_contiguous() and actions.numel() == self.n * self.j):
            a = actions                                    # fast path: already the device layout
        else:
            a = self._as_dev(actions, torch.float32, (self.n, self.j))
        self._out_buffers(write_obs, joints, final)
        if final:
            _lib.check(self._lib.mt_step_final(self._h, self._p(a), self._p(self._obs), self._p(self._reward),
                                               self._p(self._done), self._p(self._joints if joints else None),
                                               self._p(self._final.obs), self._p(self._final.episode_return),
                                               self._p(self._final.episode_length), self._stream()))
        else:
            _lib.check(self._lib.mt_step(self._h, self._p(a), self._p(self._obs if write_obs else None),
                                         self._p(self._reward), self._p(self._done),
                                         self._p(self._joints if joints else None), self._stream()))
        self._actions = a  # keep alive until the stream has consumed it
        out = (self._obs if write_obs else None, self._reward, self._done)
        if joints:
            out += (self._joints,)
        return out + (self._final,) if final else out

    def sample_actions(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Multienv.action_sample (manytor.py:111-113, 215-217): integer degrees, (N, J) f32."""
        out = out if out is not None else self._empty((self.n, self.j), torch.float32)
        _lib.check(self._lib.mt_sample_actions(self._h, self._p(out), self._stream()))
        return out

    def rollout_random(self, n_steps: int, write_obs: bool = True):
        """n_steps x step(action_sample()) with in-kernel actions; returns the last step's outputs."""
        self._out_buffers(write_obs)
        _lib.check(self._lib.mt_rollout_random(self._h, int(n_steps), self._p(self._obs if write_obs else None),
                                               self._p(self._reward), self._p(self._done), self._stream()))
        return (self._obs if write_obs else None, self._reward, self._done)

    def _check_final(self, write_obs: bool):
        if not write_obs:
            raise ValueError("final=True needs write_obs=True: the final observation is the step's obs2")
        if not self.cfg.auto_reset:
            raise ValueError("final=True needs a handle created with auto_reset=True (without auto-reset the "
                             "returned obs is the final observation and get_state() holds the return and length)")

    def _check_out(self, out, kind, arg, want, flags):
        """Validate a preallocated `out` / `final_out` namedtuple against want = {field: (shape, dtype) or None}."""
        if not isinstance(out, kind):
            raise ValueError(f"{arg} must be a {kind.__name__}")
        for name, spec in want.items():
            t = getattr(out, name)
            if spec is None:
                if t is not None:
                    raise ValueError(f"{arg}.{name} must be None here ({flags})")
                continue
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"{arg}.{name} must be a tensor of shape {spec[0]} and dtype {spec[1]}")
            if tuple(t.shape) != spec[0] or t.dtype != spec[1]:
                raise ValueError(f"{arg}.{name} must have shape {spec[0]} and dtype {spec[1]}, "
                                 f"not {tuple(t.shape)} {t.dtype}")
            if not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"{arg}.{name} must be a contiguous tensor on {self.device}")

    def rollout(self, actions=None, n_steps: Optional[int] = None, write_obs: bool = True,
                record_actions: bool = False, out: Optional[Trajectory] = None, final: bool = False,
                final_out: Optional[FinalInfo] = None):
        """K steps in one call, keeping every step: slice s of the returned Trajectory is what the s-th of K
        consecutive `step` calls would have returned, bit for bit (mt_rollout).

        actions: (K, N, J) degrees, converted like `step`'s input; K comes from it.  None = actions drawn
        in-kernel (the stream of `rollout_random` / `sample_actions`); `n_steps` then gives K, and
        `record_actions=True` returns the drawn actions as well.  `out`: a Trajectory of preallocated buffers
        (obs of this handle's obs_dtype, or None when write_obs is False; actions only with record_actions),
        e.g. fixed storage for a CUDA graph that captures this call.  Shape and dtype errors raise ValueError
        before the library is called.

        final=True (mt_rollout_final; needs auto_reset and write_obs) returns (Trajectory, FinalInfo): slice s of
        the FinalInfo holds, in the rows where done[s] != 0, what `step(final=True)` would have returned at step s
        -- the last observation ((K, N, 3X)), return and length ((K, N)) of every episode that ended there.  Other
        rows keep their contents.  `final_out`: a FinalInfo of preallocated buffers, checked like `out`."""
        if final:
            self._check_final(write_obs)
        elif final_out is not None:
            raise ValueError("final_out needs final=True")
        if actions is not None:
            if record_actions:
                raise ValueError("record_actions records in-kernel draws: it cannot be combined with actions")
            shape = tuple(actions.shape) if hasattr(actions, "shape") else tuple(np.shape(actions))
            if len(shape) != 3 or shape[1:] != (self.n, self.j):
                raise ValueError(f"actions must have shape (K, {self.n}, {self.j}), not {shape}")
            if n_steps is not None and int(n_steps) != shape[0]:
                raise ValueError(f"n_steps={n_steps} disagrees with the {shape[0]} steps of actions")
            k = shape[0]
        else:
            if n_steps is None:
                raise ValueError("rollout needs actions or n_steps")
            k = int(n_steps)
        if k < 0:
            raise ValueError(f"n_steps must be >= 0, not {k}")
        want = {"obs": ((k, self.n, 3 * self.x), self.obs_dtype) if write_obs else None,
                "reward": ((k, self.n), torch.float32), "done": ((k, self.n), torch.uint8),
                "actions": ((k, self.n, self.j), torch.float32) if record_actions else None}
        if out is not None:
            self._check_out(out, Trajectory, "out", want, f"write_obs={write_obs}, record_actions={record_actions}")
            bufs = out
        else:
            bufs = Trajectory(*(self._empty(*spec) if spec is not None else None for spec in want.values()))
        fin = None
        if final:
            want_fin = {"obs": ((k, self.n, 3 * self.x), self.obs_dtype), "episode_return": ((k, self.n), torch.float32),
                        "episode_length": ((k, self.n), torch.int32)}
            if final_out is not None:
                self._check_out(final_out, FinalInfo, "final_out", want_fin, "")
                fin = final_out
            else:
                fin = FinalInfo(*(self._empty(*spec) for spec in want_fin.values()))
        if actions is not None:
            if (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.device == self.device
                    and actions.dtype == torch.float32 and actions.is_contiguous()):
                a = actions                                # fast path: already the device layout
            else:
                a = self._as_dev(actions, torch.float32, (k, self.n, self.j))
            bufs = bufs._replace(actions=a)
        if k == 0:                                         # nothing to do (and empty tensors have no address)
            return (bufs, fin) if final else bufs
        a_p, d_p = self._p(a if actions is not None else None), self._p(bufs.actions if actions is None else None)
        if final:
            _lib.check(self._lib.mt_rollout_final(self._h, k, a_p, d_p, self._p(bufs.obs), self._p(bufs.reward),
                                                  self._p(bufs.done), self._p(fin.obs), self._p(fin.episode_return),
                                                  self._p(fin.episode_length), self._stream()))
        else:
            _lib.check(self._lib.mt_rollout(self._h, k, a_p, d_p, self._p(bufs.obs), self._p(bufs.reward),
                                            self._p(bufs.done), self._stream()))
        self._rollout_io = (bufs, fin)                     # keep alive until the stream has consumed them
        return (bufs, fin) if final else bufs

    def rollout_branches(self, actions, src=None, gamma: float = 1.0, write_obs: bool = False,
                         out: Optional[Branches] = None, *, n_steps: Optional[int] = None, draw_key=None) -> Branches:
        """Score K-step action sequences from copies of chosen envs in one launch, leaving this handle untouched
        (mt_rollout_branches): branch m starts from the current state of env src[m] and steps with actions[:, m] as
        `step` would, until its first done step (included) or the K-th step.  No env is reset inside a branch, and the
        state, objectives, reset counts, statistics and step index of the handle stay as they were.

        actions: (K, M, J) degrees, converted like `rollout`'s input.  src: (M,) integers, the source env of each branch
        (repeats and any order allowed); a tensor on this device is used as it is, without a host synchronisation.
        None means arange(N), which needs M == N.  A source outside [0, N) gives that branch ret NaN, length -1, done 0
        and leaves its obs row alone.  gamma in [0, 1]: ret is sum of gamma**s * r_s in fp32, d_0 = 1, d_{s+1} = d_s *
        gamma, G += d_s * r_s.  write_obs: also return obs2 of each branch's last executed step.  `out`: a Branches of
        preallocated buffers (obs None unless write_obs), e.g. fixed storage for a CUDA graph that captures this call.
        Shape and dtype errors raise ValueError before the library is called.

        In-kernel draws (mt_rollout_branches_random), with `n_steps` and / or `draw_key`: the branches run n_steps = K
        steps (default: the prefix's length; required without a prefix); `actions` is None (every step drawn) or a
        (P, M, J) prefix of the first P <= K steps, and the other steps take the environment's own random policy,
        integer degrees uniform on [action_low, action_high).  Step s of branch m draws what `sample_actions` draws for global env id m at step
        index draw_key + s (mod 2^64): the draws depend on (seed, m, draw_key) only, and `branch_actions` returns them
        again.  Calls whose [draw_key, draw_key + K) overlap reuse draws, so advance the key by K per call.  draw_key:
        an int, or a (1,) int64 tensor on this device holding the key's bits, read by the kernel (a CUDA graph that
        captures this call and a `key += K` draws fresh actions at every replay).  M is len(src), or N with src=None."""
        if n_steps is not None or draw_key is not None:
            return self._rollout_branches_random(actions, src, gamma, write_obs, out, n_steps, draw_key)
        shape = tuple(actions.shape) if hasattr(actions, "shape") else tuple(np.shape(actions))
        if len(shape) != 3 or shape[2] != self.j:
            raise ValueError(f"actions must have shape (K, M, {self.j}), not {shape}")
        k, m = shape[0], shape[1]
        if k > 4096:
            raise ValueError(f"rollout_branches takes at most 4096 steps, not {k}")
        g = float(gamma)
        if not 0.0 <= g <= 1.0:
            raise ValueError(f"gamma must be finite and in [0, 1], not {gamma}")
        if src is None:
            if m != self.n:
                raise ValueError(f"src=None branches every env once: actions need M = {self.n} branches, not {m}")
        else:
            src_shape = tuple(src.shape) if hasattr(src, "shape") else tuple(np.shape(src))
            if src_shape != (m,):
                raise ValueError(f"src must have shape ({m},) (one source per branch), not {src_shape}")
            src_dtype = src.dtype if isinstance(src, torch.Tensor) else torch.as_tensor(np.asarray(src)).dtype
            if src_dtype.is_floating_point or src_dtype.is_complex or src_dtype == torch.bool:
                raise ValueError(f"src must hold integers, not {src_dtype}")
        want = {"ret": ((m,), torch.float32), "length": ((m,), torch.int32), "done": ((m,), torch.uint8),
                "obs": ((m, 3 * self.x), self.obs_dtype) if write_obs else None}
        if out is not None:
            self._check_out(out, Branches, "out", want, f"write_obs={write_obs}")
            bufs = out
        else:
            bufs = Branches(*(self._empty(*spec) if spec is not None else None for spec in want.values()))
        if k == 0 or m == 0:                               # nothing to do (and empty tensors have no address)
            return bufs
        if (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.device == self.device
                and actions.dtype == torch.float32 and actions.is_contiguous()):
            a = actions                                    # fast path: already the device layout
        else:
            a = self._as_dev(actions, torch.float32, (k, m, self.j))
        if src is None:
            s = torch.arange(self.n, dtype=torch.int64, device=self.device)
        elif (isinstance(src, torch.Tensor) and src.is_cuda and src.device == self.device and src.dtype == torch.int64
                and src.is_contiguous()):
            s = src
        else:
            s = self._as_dev(src, torch.int64, (m,))
        _lib.check(self._lib.mt_rollout_branches(self._h, k, m, self._p(s), self._p(a), g, self._p(bufs.ret),
                                                 self._p(bufs.length), self._p(bufs.done), self._p(bufs.obs),
                                                 self._stream()))
        self._branch_io = (a, s, bufs)                     # keep alive until the stream has consumed them
        return bufs

    def _draw_key(self, draw_key, check_only: bool = False):
        """The device word of a draw key: a (1,) int64 tensor on this device as it is, or an int (mod 2^64) in a fresh
        one-element tensor of its own, so that no later call, on whatever stream, can overwrite it before it is read."""
        if isinstance(draw_key, torch.Tensor):
            if tuple(draw_key.shape) != (1,) or draw_key.dtype != torch.int64 or draw_key.device != self.device:
                raise ValueError(f"draw_key must be an int or a (1,) int64 tensor on {self.device}, not a "
                                 f"{tuple(draw_key.shape)} {draw_key.dtype} tensor on {draw_key.device}")
            return draw_key
        if isinstance(draw_key, (bool, np.bool_)) or not isinstance(draw_key, (int, np.integer)):
            raise ValueError(f"draw_key must be an int or a (1,) int64 tensor on {self.device}, not {draw_key!r}")
        if check_only:
            return None
        k = int(draw_key) % (1 << 64)
        return torch.full((1,), k - (1 << 64) if k >= 1 << 63 else k, dtype=torch.int64, device=self.device)

    def _aligned_dev(self, a, dtype, shape) -> torch.Tensor:
        """`a` as a contiguous device tensor of `dtype` and `shape` whose address is 16-byte aligned, as the library
        requires: such a tensor on this device as it is, anything else converted, and a view that starts off the
        alignment (e.g. best[1:]) copied into storage of its own."""
        if (isinstance(a, torch.Tensor) and a.is_cuda and a.device == self.device and a.dtype == dtype
                and a.is_contiguous() and a.data_ptr() % 16 == 0):
            return a.reshape(shape)
        t = self._as_dev(a, dtype, shape)
        return t if t.data_ptr() % 16 == 0 else t.clone()

    def _dev_ids(self, ids, m: int) -> torch.Tensor:
        """(m,) integers as an int64 device tensor (_aligned_dev)."""
        return self._aligned_dev(ids, torch.int64, (m,))

    @staticmethod
    def _int_vector(v, name: str, m: Optional[int] = None) -> int:
        """Check that v is a 1-D array of integers (of m entries when m is given); return its length."""
        shape = tuple(v.shape) if hasattr(v, "shape") else tuple(np.shape(v))
        if len(shape) != 1 or (m is not None and shape[0] != m):
            raise ValueError(f"{name} must have shape ({'M' if m is None else m},), not {shape}")
        dtype = v.dtype if isinstance(v, torch.Tensor) else torch.as_tensor(np.asarray(v)).dtype
        if dtype.is_floating_point or dtype.is_complex or dtype == torch.bool:
            raise ValueError(f"{name} must hold integers, not {dtype}")
        return shape[0]

    def _rollout_branches_random(self, actions, src, gamma, write_obs, out, n_steps, draw_key) -> Branches:
        if draw_key is None:
            raise ValueError("in-kernel draws need an explicit draw_key: the same key regenerates them (branch_actions)")
        self._draw_key(draw_key, check_only=True)
        m = self.n if src is None else self._int_vector(src, "src")
        p = 0
        if actions is not None:
            shape = tuple(actions.shape) if hasattr(actions, "shape") else tuple(np.shape(actions))
            if len(shape) != 3 or shape[1:] != (m, self.j):
                raise ValueError(f"a prefix of actions must have shape (P, {m}, {self.j}) (M = "
                                 f"{'N' if src is None else 'len(src)'}), not {shape}")
            p = shape[0]
        if n_steps is None and actions is None:
            raise ValueError("n_steps is required when actions is None (every step drawn): it is the branches' length")
        k = p if n_steps is None else int(n_steps)
        if not 0 <= k <= 4096:
            raise ValueError(f"n_steps must be in [0, 4096], not {k}")
        if p > k:
            raise ValueError(f"the prefix has {p} steps, more than n_steps = {k}")
        g = float(gamma)
        if not 0.0 <= g <= 1.0:
            raise ValueError(f"gamma must be finite and in [0, 1], not {gamma}")
        want = {"ret": ((m,), torch.float32), "length": ((m,), torch.int32), "done": ((m,), torch.uint8),
                "obs": ((m, 3 * self.x), self.obs_dtype) if write_obs else None}
        if out is not None:
            self._check_out(out, Branches, "out", want, f"write_obs={write_obs}")
            bufs = out
        else:
            bufs = Branches(*(self._empty(*spec) if spec is not None else None for spec in want.values()))
        if k == 0 or m == 0:                               # nothing to do (and empty tensors have no address)
            return bufs
        a = self._aligned_dev(actions, torch.float32, (p, m, self.j)) if p > 0 else None
        s = torch.arange(self.n, dtype=torch.int64, device=self.device) if src is None else self._dev_ids(src, m)
        key = self._draw_key(draw_key)
        _lib.check(self._lib.mt_rollout_branches_random(self._h, k, p, m, self._p(s), self._p(a), self._p(key), g,
                                                        self._p(bufs.ret), self._p(bufs.length), self._p(bufs.done),
                                                        self._p(bufs.obs), self._stream()))
        self._branch_io = (a, s, key, bufs)                # keep alive until the stream has consumed them
        return bufs

    def branch_actions(self, branches, draw_key, n_steps: int, first_step: int = 0,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The actions in-kernel draws give chosen branches (mt_branch_actions): out[s, r] = the actions of branch id
        branches[r] at branch step first_step + s under `draw_key`, as `rollout_branches(draw_key=...)` drew them --
        `sample_actions` for global env id branches[r] at step index draw_key + first_step + s (mod 2^64).  Returns
        (n_steps, R, J) float32.  The action a planner executes after picking branch b: branch_actions([b], key, 1).
        branches: (R,) integers, any int64 value.  draw_key: as in rollout_branches.  Needs no reset and changes nothing
        of the handle.  Shape and range errors raise ValueError before the library is called."""
        r = self._int_vector(branches, "branches")
        self._draw_key(draw_key, check_only=True)
        k, first = int(n_steps), int(first_step)
        if not 0 <= k < 1 << 31:
            raise ValueError(f"n_steps must be in [0, 2^31), not {n_steps}")
        if not 0 <= first < 1 << 31:
            raise ValueError(f"first_step must be in [0, 2^31), not {first_step}")
        if r > 2000000000:
            raise ValueError(f"at most 2000000000 branches, not {r}")
        shape = (k, r, self.j)
        if out is None:
            out = self._empty(shape, torch.float32)
        elif not isinstance(out, torch.Tensor) or tuple(out.shape) != shape or out.dtype != torch.float32:
            raise ValueError(f"out must be a tensor of shape {shape} and dtype torch.float32")
        elif not out.is_contiguous() or out.device != self.device or out.data_ptr() % 16 != 0:
            raise ValueError(f"out must be a contiguous, 16-byte aligned tensor on {self.device}")
        if k == 0 or r == 0:                               # nothing to do (and empty tensors have no address)
            return out
        ids, key = self._dev_ids(branches, r), self._draw_key(draw_key)
        _lib.check(self._lib.mt_branch_actions(self._h, self._p(key), first, k, r, self._p(ids), self._p(out),
                                               self._stream()))
        self._branch_actions_io = (ids, key, out)          # keep alive until the stream has consumed them
        return out

    # -- host-buffer (end-to-end) step ------------------------------------------
    def pinned(self, name: str, shape, dtype) -> np.ndarray:
        key = (name, tuple(shape), np.dtype(dtype).str)
        if key not in self._pinned:
            pa = self._pinned[key] = PinnedArray(shape, dtype)
            self._pinned_ptr[id(pa.array)] = pa.ptr
        return self._pinned[key].array

    def step_host(self, actions_host: np.ndarray, write_obs: bool = True):
        """Step with HOST buffers: H2D(actions) + kernel + D2H(obs, reward, done), chunked
        and overlapped on internal streams.  `actions_host` should come from
        `pinned(name, (N, J), float32)` (any name: several buffers can be cycled); other
        input is staged through `pinned('actions', ...)`.  The returned arrays are views of
        page-locked buffers that the NEXT step_host overwrites; they stay valid (they own the
        allocation) even after this object is gone."""
        io = self._host_io.get(write_obs)
        if io is None:                                     # buffers and addresses once: a batch of one is pure latency
            act = self.pinned("actions", (self.n, self.j), np.float32)
            obs_np = np.float16 if self.obs_dtype == torch.float16 else np.float32
            obs = self.pinned("obs", (self.n, 3 * self.x), obs_np) if write_obs else None
            rew = self.pinned("reward", (self.n,), np.float32)
            done = self.pinned("done", (self.n,), np.uint8)
            addr = lambda a: self._pinned_ptr[id(a)] if a is not None else None
            io = self._host_io[write_obs] = (act, addr(act), obs, addr(obs), rew, addr(rew), done, addr(done))
        act, act_ptr, obs, obs_ptr, rew, rew_ptr, done, done_ptr = io
        own = self._pinned_ptr.get(id(actions_host))       # already one of this object's page-locked buffers?
        if own is None:
            np.copyto(act, np.asarray(actions_host, dtype=np.float32).reshape(self.n, self.j))
            own = act_ptr
        self._after_side_stream()
        _lib.check(self._lib.mt_step_host(self._h, own, obs_ptr, rew_ptr, done_ptr))
        return obs, rew, done

    @property
    def host_step_mode(self) -> str:
        """Which implementation `step_host` settled on for this handle (it times both on its first calls)."""
        return {0: "staged", 1: "zero-copy", 2: "deciding"}.get(int(self._lib.mt_host_step_mode(self._h)), "?")

    # -- state exchange ---------------------------------------------------------
    def set_points(self, points, mask=None):
        p = self._as_dev(points, torch.float32, (self.n, self.x, 3))
        _lib.check(self._lib.mt_set_points(self._h, self._p(p), self._p(self._mask(mask)), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def get_points(self, zero_dead: bool = True) -> torch.Tensor:
        out = self._empty((self.n, self.x, 3), torch.float32)
        _lib.check(self._lib.mt_get_points(self._h, self._p(out), int(zero_dead), self._stream()))
        return out

    def set_state(self, goals=None, alive=None, total_reward=None, ep_len=None, mask=None, resets=None):
        """Overwrite parts of the state (None = keep).  `resets`: (N,) per-env reset counts, integers whose low 32 bits
        are the uint32 count (the int32 `get_state()["resets"]` as it is).  Restoring a checkpoint: see get_state."""
        if resets is not None and tuple(np.shape(resets)) != (self.n,):
            raise ValueError(f"resets must have shape ({self.n},), not {tuple(np.shape(resets))}")
        g = self._as_dev(goals, torch.float32, (self.n, self.j)) if goals is not None else None
        al = self._alive_words(alive) if alive is not None else None
        tr = self._as_dev(total_reward, torch.float32, (self.n,)) if total_reward is not None else None
        el = self._as_dev(ep_len, torch.int32, (self.n,)) if ep_len is not None else None
        m = self._mask(mask)
        _lib.check(self._lib.mt_set_state(self._h, self._p(g), self._p(al), self._p(tr), self._p(el),
                                          self._p(m), self._stream()))
        if resets is not None:
            rc = self._u32_words(resets)
            _lib.check(self._lib.mt_set_reset_counts(self._h, self._p(rc), self._p(m), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def _alive_words(self, alive) -> torch.Tensor:
        """(N, X) bool or (N,) integer bitmask -> (N,) int32 holding the uint32 bit pattern."""
        al = torch.as_tensor(alive)
        if al.dim() == 2:
            w = (1 << torch.arange(self.x, dtype=torch.int64))
            al = (al.to(torch.int64) * w).sum(dim=1)
        return self._u32_words(al)

    def _u32_words(self, words) -> torch.Tensor:
        """(N,) integers -> (N,) int32 on the device holding their low 32 bits (the uint32 bit pattern)."""
        w = torch.as_tensor(words).to(torch.int64) & 0xFFFFFFFF
        w = torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)
        return w.to(self.device).contiguous().reshape(self.n)

    def get_state(self) -> dict:
        """goals (N, J) f32, alive (N,) int32 holding the uint32 bitmask, total_reward (N,) f32, ep_len (N,) int32 and
        resets (N,) int32 holding each env's uint32 reset count (it keys the objective sampler and picks the objective
        stream's set).  With raw points (get_points(zero_dead=False)) and step_index this is what a handle created with
        the same config (and objective stream) needs to continue bit for bit: reset() it, then set_state(**state),
        set_points and step_index.  Statistics are not part of it: the new handle counts from zero."""
        g = self._empty((self.n, self.j), torch.float32)
        al = self._empty((self.n,), torch.int32)
        tr = self._empty((self.n,), torch.float32)
        el = self._empty((self.n,), torch.int32)
        rc = self._empty((self.n,), torch.int32)
        _lib.check(self._lib.mt_get_state(self._h, self._p(g), self._p(al), self._p(tr), self._p(el), self._stream()))
        _lib.check(self._lib.mt_get_reset_counts(self._h, self._p(rc), self._stream()))
        return dict(goals=g, alive=al, total_reward=tr, ep_len=el, resets=rc)

    def alive_matrix(self) -> torch.Tensor:
        """(N, X) bool view of the alive bitmask (the reference's `alives`, manytor.py:134)."""
        al = self.get_state()["alive"].to(torch.int64) & 0xFFFFFFFF
        bits = torch.arange(self.x, device=self.device, dtype=torch.int64)
        return ((al[:, None] >> bits[None, :]) & 1).bool()

    def set_objective_stream(self, points):
        """points (E, N, X, 3): the e-th reset of env n takes set e mod E (parity runs)."""
        if points is None:
            _lib.check(self._lib.mt_set_objective_stream(self._h, None, 0))
            self._stream_keepalive = None
            return
        p = self._as_dev(points, torch.float32)
        assert p.dim() == 4 and tuple(p.shape[1:]) == (self.n, self.x, 3), p.shape
        torch.cuda.current_stream(self.device).synchronize()
        _lib.check(self._lib.mt_set_objective_stream(self._h, self._p(p), int(p.shape[0])))
        self._stream_keepalive = p

    def joints_of(self, goals) -> torch.Tensor:
        """joints_coordinates (manytor.py:188-189) of arbitrary poses (M, J) -> (M, J, 3)."""
        g = self._as_dev(goals, torch.float32).reshape(-1, self.j)
        out = self._empty((g.shape[0], self.j, 3), torch.float32)
        _lib.check(self._lib.mt_joints(self._h, self._p(g), self._p(out), g.shape[0], self._stream()))
        return out

    def fetch_env(self, index: int) -> dict:
        """One-env copy-back for rendering / attribute access (manytor.py:131-139)."""
        goals = np.zeros(self.j, dtype=np.float32)
        joints = np.zeros((self.j, 3), dtype=np.float32)
        points = np.zeros((self.x, 3), dtype=np.float32)
        alive = C.c_uint32()
        total = C.c_float()
        self._after_side_stream()
        _lib.check(self._lib.mt_fetch_env(self._h, int(index), goals.ctypes.data, joints.ctypes.data,
                                          points.ctypes.data, C.byref(alive), C.byref(total)))
        alives = np.array([(alive.value >> p) & 1 for p in range(self.x)], dtype=bool)
        return dict(goals=goals, joints_coordinates=joints, points=points, alives=alives,
                    total_reward=float(total.value))

    def set_seed(self, seed: int):
        """Re-seed the on-device action / objective streams (gym-style reset(seed=...)): new Philox key,
        per-env episode counters and the step index back to zero, so the same seed reproduces the same
        objectives and actions on the same handle."""
        _lib.check(self._lib.mt_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF))
        self.cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF

    @property
    def step_index(self) -> int:
        """Steps executed so far; keys the action stream.  Lives on the device (advanced by the step
        kernel, so CUDA-graph replays count); reading it synchronises."""
        v = C.c_uint64()
        self._after_side_stream()
        _lib.check(self._lib.mt_get_step_index(self._h, C.byref(v)))
        return int(v.value)

    @step_index.setter
    def step_index(self, value: int):
        """Resume from a checkpoint.  Accepts [0, 2^62] (MT_STEP_INDEX_MAX); anything else raises ValueError."""
        value = int(value)
        if not 0 <= value <= _lib.MT_STEP_INDEX_MAX:
            raise ValueError(f"step_index must be in [0, 2**62], not {value}")
        self._after_side_stream()
        _lib.check(self._lib.mt_set_step_index(self._h, value))

    # -- statistics ---------------------------------------------------------------
    def stats_tensor(self) -> torch.Tensor:
        """MT_STATS_WORDS int64 on the device (sum-reducible across shards)."""
        out = self._empty((_lib.MT_STATS_WORDS,), torch.int64)
        _lib.check(self._lib.mt_stats_device(self._h, self._p(out), self._stream()))
        return out

    def stats(self) -> dict:
        s = MtStats()
        self._after_side_stream()
        _lib.check(self._lib.mt_stats_host(self._h, C.byref(s)))
        return {k: int(getattr(s, k)) for k in STATS_FIELDS}

    def clear_stats(self):
        _lib.check(self._lib.mt_stats_clear(self._h, self._stream()))

    # -- introspection --------------------------------------------------------------
    @property
    def launch_count(self) -> int:
        return int(self._lib.mt_launch_count(self._h))

    def bytes_per_env_step(self, actions_from_hbm: bool = True, obs_written: bool = True) -> int:
        return int(self._lib.mt_bytes_per_env_step(self._h, int(actions_from_hbm), int(obs_written)))

    def set_timing(self, enabled: bool):
        _lib.check(self._lib.mt_set_timing(self._h, int(enabled)))

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        _lib.check(self._lib.mt_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)
