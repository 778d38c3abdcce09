"""Gymnasium-style vector environment over the batched CUDA step loop (SURVEY.md section 8f).

The reference's API is the gym-like 3-tuple of manytor.py:255-260; RL libraries today expect the
Gymnasium vector-env convention instead:

    obs, info = env.reset(seed=...)
    obs, reward, terminated, truncated, info = env.step(actions)

This adapter provides exactly that on DEVICE tensors (nothing is copied to the host): `obs` is a
torch view of the buffer the step kernel wrote (row-major (N, 3X), fp32 or, with obs_dtype=torch.float16,
binary16 written by the kernel itself), so a policy network on the
same GPU consumes it directly; `torch.utils.dlpack.to_dlpack(obs)` / `obs.__dlpack__()` hands the
same memory to JAX/CuPy without a copy.  Auto-reset is "same-step": an env that terminates
(all objectives collected, manytor.py:170-171) or is truncated (horizon reached, the `max_steps` of
the reference's driver scripts) is reset inside the step kernel and the observation returned for it
is the FIRST observation of its next episode.

With `final_info=True` the observation that closed the episode (obs2 of the ending step, which a
truncated episode needs to bootstrap its return from V(final_obs)) and the episode's return and length
come back in `info`, written by the same kernel (mt_step_final), as device tensors:

    {"final_obs": (N, 3X), "_final_obs": terminated | truncated,
     "episode": {"r": (N,) float32, "l": (N,) int32}, "_episode": terminated | truncated}

Rows outside the masks are unspecified.  With the default `final_info=False` that observation, return
and length are gone after the step and `info` is empty.  No gymnasium import is needed; the space
attributes are plain shape/bound tuples.
"""
from __future__ import annotations

from typing import Optional

import torch

from .core import ArmSpec, BatchedEnvs, REFERENCE_ARM


class ManyTorVectorEnv:
    metadata = {"autoreset_mode": "same_step"}

    def __init__(self, num_envs: int, obj_number: int = 10, arm: ArmSpec = REFERENCE_ARM, max_episode_steps: int = 200,
                 device=None, seed: int = 0, terminate_on_ground: bool = False, env_id_base: int = 0,
                 obs_dtype=torch.float32, final_info: bool = False):
        self.num_envs = int(num_envs)
        self.final_info = bool(final_info)
        self.envs = BatchedEnvs(num_envs, obj_number, arm=arm, device=device, env_id_base=env_id_base,
                                horizon=max_episode_steps, auto_reset=True, obs_after_reset=True,
                                terminate_on_ground=terminate_on_ground, seed=seed, obs_dtype=obs_dtype)
        self.single_observation_shape = (3 * obj_number,)
        self.single_action_shape = (arm.n_joints,)
        self.action_low, self.action_high = -180.0, 180.0            # degrees, manytor.py:216
        self.observation_shape = (self.num_envs,) + self.single_observation_shape
        self.action_shape = (self.num_envs,) + self.single_action_shape
        self.device = self.envs.device

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        if seed is not None:
            self.envs.set_seed(seed)
        obs = self.envs.reset(returnable=True)
        return obs, {}

    def step(self, actions):
        if self.final_info:
            obs, reward, done, final = self.envs.step(actions, final=True)
        else:
            obs, reward, done = self.envs.step(actions)
        terminated = (done & 1).bool()
        truncated = (done & 2).bool()
        if not self.final_info:
            return obs, reward, terminated, truncated, {}
        ended = terminated | truncated
        info = {"final_obs": final.obs, "_final_obs": ended,
                "episode": {"r": final.episode_return, "l": final.episode_length}, "_episode": ended}
        return obs, reward, terminated, truncated, info

    def sample_actions(self) -> torch.Tensor:
        """Uniform integer-degree actions like `action_sample()` (manytor.py:215-217), on device."""
        return self.envs.sample_actions()

    def episode_statistics(self) -> dict:
        return self.envs.stats()

    def close(self):
        self.envs.close()
