"""NoiseObservationWrapper (tinycarlo/wrapper/observation.py:5-33): random blob noise on class masks — filled circles that
erase a class mask or OR in the pixels of a random class — as a device kernel (tc_noise_blobs) for the vectorised env and
for the single-env drop-in. Same constructor arguments as the reference plus `seed`: the reference draws from numpy's
unseeded global RNG, so there is no stream to reproduce; here the noise of (env, step, class, blob) is a pure function of
the seed through Philox4x32-10 (contract in include/tinycarlo_b200.h), reproducible and independent of the GPU sharding.
With a camera rig every view is noised: camera m draws with counter word 3 = m, so camera 0 gets the rig-less noise. On a
TinyCarloGroupedVecEnv each group's observation is noised with its own handle and env_index_offset, so the noise of an env
depends on its global index only. Like the reference, constructing it sets `unwrapped.wrapped = True` and it only acts
on the "classes" format."""
import ctypes as C

import torch

from .. import _lib
from ..grouped_env import TinyCarloGroupedVecEnv
from ..gym_compat import Wrapper
from .reward import _VecWrapper, _make


def _apply(vec, obs: torch.Tensor, seed: int, step: int, n_blobs: int, max_radius: int):
    with torch.cuda.device(vec.device):
        _lib.check(vec._L.tc_noise_blobs(vec._h, C.c_void_p(obs.data_ptr()), int(seed) & (2**64 - 1), int(step) & 0xFFFFFFFF, int(n_blobs),
                                         int(max_radius), int(vec.env_index_offset), None,
                                         C.c_void_p(torch.cuda.current_stream(vec.device).cuda_stream)), "tc_noise_blobs")


class _NoiseVec(_VecWrapper):
    def __init__(self, env, blob_max_radius=100, n_blobs=10, seed=0):
        super().__init__(env)
        self.max_radius, self.n_blobs, self.seed = blob_max_radius, n_blobs, seed
        self.steps = 0

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        u = self.unwrapped
        # a grouped env returns one observation tensor per group, each owned by that group's env
        for e, obs in zip(u.envs, observation) if isinstance(u, TinyCarloGroupedVecEnv) else [(u, observation)]:
            if e.observation_space_format == "classes" and not e.no_observation:
                _apply(e, obs, self.seed, self.steps, self.n_blobs, self.max_radius)   # in place, like the reference
        self.steps += 1
        return observation, reward, terminated, truncated, info


class _NoiseScalar(Wrapper):
    def __init__(self, env, blob_max_radius=100, n_blobs=10, seed=0):
        super().__init__(env)
        self.unwrapped.wrapped = True
        self.max_radius, self.n_blobs, self.seed = blob_max_radius, n_blobs, seed
        self.steps = 0

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        u = self.env.unwrapped
        if u.observation_space_format == "classes" and not u.no_observation:
            vec = u._vec
            _apply(vec, vec.obs, self.seed, self.steps, self.n_blobs, self.max_radius)
            observation = vec.obs[0].cpu().numpy().copy()
        self.steps += 1
        return observation, reward, terminated, truncated, info


class NoiseObservationWrapper:
    """NoiseObservationWrapper(env, blob_max_radius=100, n_blobs=10, seed=0)"""
    __new__ = _make(_NoiseScalar, _NoiseVec)


for _i in (_NoiseScalar, _NoiseVec):
    _i.__name__ = "NoiseObservationWrapper"
