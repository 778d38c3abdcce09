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
is the FIRST observation of its next episode.  No gymnasium import is needed; the space attributes
are plain shape/bound tuples.
"""
from __future__ import annotations

from typing import Optional

import torch

from .core import ArmSpec, BatchedEnvs, REFERENCE_ARM


class ManyTorVectorEnv:
    metadata = {"autoreset_mode": "same_step"}

    def __init__(self, num_envs: int, obj_number: int = 10, arm: ArmSpec = REFERENCE_ARM, max_episode_steps: int = 200,
                 device=None, seed: int = 0, terminate_on_ground: bool = False, env_id_base: int = 0,
                 obs_dtype=torch.float32):
        self.num_envs = int(num_envs)
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
        obs, reward, done = self.envs.step(actions)
        terminated = (done & 1).bool()
        truncated = (done & 2).bool()
        return obs, reward, terminated, truncated, {}

    def sample_actions(self) -> torch.Tensor:
        """Uniform integer-degree actions like `action_sample()` (manytor.py:215-217), on device."""
        return self.envs.sample_actions()

    def episode_statistics(self) -> dict:
        return self.envs.stats()

    def close(self):
        self.envs.close()
