"""Reward wrappers with the reference's names, arguments and arithmetic (tinycarlo/wrapper/reward.py:5-84). Each class
wraps either the single-env drop-in (gymnasium-style Wrapper, Python scalars) or a TinyCarloVecEnv (tensor ops on the
device, no host sync), chosen by what is passed in. Constructing one sets `unwrapped.wrapped = True`, which switches the
default reward/termination of the env off (env.py:137-138)."""
from typing import Dict

import torch

from ..gym_compat import Wrapper
from .utils import linear_reward, linear_reward_tensor, sparse_reward


def _is_vec(env) -> bool:
    return getattr(env, "is_vector_env", False) or getattr(getattr(env, "unwrapped", None), "is_vector_env", False)


class _VecWrapper:
    """Minimal wrapper base for the vectorised env (it is not a gymnasium Env)."""
    is_vector_env = True

    def __init__(self, env):
        self.env = env
        self.unwrapped.set_wrapped(True)

    @property
    def unwrapped(self):
        return getattr(self.env, "unwrapped", self.env)

    def __getattr__(self, name):
        if name == "env":
            raise AttributeError(name)
        return getattr(self.env, name)

    def reset(self, *a, **kw):
        return self.env.reset(*a, **kw)

    def reset_done(self):
        return self.env.reset_done()

    def step(self, action):
        return self.env.step(action)

    def _live(self, bonus: torch.Tensor) -> torch.Tensor:
        """the wrapper's reward term, zero for envs that this step autoreset (no transition happened: gymnasium's
        next-step autoreset returns reward 0 there, and a caller of the reference would have called reset() instead)"""
        u = self.unwrapped
        if getattr(u, "autoreset", None):
            return torch.where(u.reset_mask, torch.zeros_like(bonus), bonus)
        return bonus


def _make(cls_scalar, cls_vec):
    """class factory: Name(env, ...) -> scalar or vector implementation"""
    def new(cls, env, *a, **kw):
        impl = cls_vec if _is_vec(env) else cls_scalar
        obj = object.__new__(impl)
        impl.__init__(obj, env, *a, **kw)   # obj is not an instance of cls, so Python will not call __init__ itself
        return obj
    return new


# ------------------------------------------------------------------------------------------------ laneline sparse
class _LanelineSparseScalar(Wrapper):
    def __init__(self, env, sparse_rewards: Dict[str, float]):
        super().__init__(env)
        self.unwrapped.wrapped = True
        self.sparse_rewards = sparse_rewards

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        tw = self.unwrapped.car.track_width
        conditions = {n: info["laneline_distances"][n] < tw / 2 for n in info["laneline_distances"]}
        reward += sparse_reward(conditions, self.sparse_rewards)
        return observation, reward, terminated, truncated, info


class _LanelineSparseVec(_VecWrapper):
    def __init__(self, env, sparse_rewards: Dict[str, float]):
        super().__init__(env)
        self.sparse_rewards = sparse_rewards
        u = self.unwrapped
        self._w = torch.tensor([float(sparse_rewards.get(n, 0.0)) for n in u.class_names], dtype=torch.float32, device=u.device)

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        cond = info["laneline_distances"] < self.unwrapped.track_width / 2
        reward = reward + self._live((cond.to(torch.float32) * self._w).sum(dim=1))
        return observation, reward, terminated, truncated, info


class LanelineSparseRewardWrapper:
    """reward += sparse_rewards[name] for every laneline closer than track_width/2 (reward.py:5-23)."""
    __new__ = _make(_LanelineSparseScalar, _LanelineSparseVec)


# ------------------------------------------------------------------------------------------------ laneline linear
class _LanelineLinearScalar(Wrapper):
    def __init__(self, env, max_rewards: Dict[str, float]):
        super().__init__(env)
        self.unwrapped.wrapped = True
        self.max_rewards = max_rewards

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        for name, distance in info["laneline_distances"].items():
            reward += linear_reward(distance, self.unwrapped.car.track_width, self.max_rewards[name])
        return observation, reward, terminated, truncated, info


class _LanelineLinearVec(_VecWrapper):
    def __init__(self, env, max_rewards: Dict[str, float]):
        super().__init__(env)
        self.max_rewards = max_rewards
        for n in self.unwrapped.class_names:
            max_rewards[n]  # KeyError like the reference when a laneline has no entry

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        u = self.unwrapped
        for k, n in enumerate(u.class_names):
            reward = reward + self._live(linear_reward_tensor(info["laneline_distances"][:, k], u.track_width, self.max_rewards[n]))
        return observation, reward, terminated, truncated, info


class LanelineLinearRewardWrapper:
    """reward += linear_reward(distance, track_width, max_rewards[name]) per laneline (reward.py:25-42)."""
    __new__ = _make(_LanelineLinearScalar, _LanelineLinearVec)


# ------------------------------------------------------------------------------------------------ CTE sparse
class _CTESparseScalar(Wrapper):
    def __init__(self, env, min_cte: float, sparse_reward: float = 1.0):
        super().__init__(env)
        self.unwrapped.wrapped = True
        self.min_cte = min_cte
        self.sparse_reward = sparse_reward

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        reward += sparse_reward({"cte": abs(info["cte"]) <= self.min_cte}, {"cte": self.sparse_reward})
        return observation, reward, terminated, truncated, info


class _CTESparseVec(_VecWrapper):
    def __init__(self, env, min_cte: float, sparse_reward: float = 1.0):
        super().__init__(env)
        self.min_cte = min_cte
        self.sparse_reward = sparse_reward

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        reward = reward + self._live((info["cte"].abs() <= self.min_cte).to(torch.float32) * self.sparse_reward)
        return observation, reward, terminated, truncated, info


class CTESparseRewardWrapper:
    """reward += sparse_reward when |cte| <= min_cte (reward.py:44-62)."""
    __new__ = _make(_CTESparseScalar, _CTESparseVec)


# ------------------------------------------------------------------------------------------------ CTE linear
class _CTELinearScalar(Wrapper):
    def __init__(self, env, min_cte: float, max_reward: float = 1.0, min_reward: float = 0.0):
        super().__init__(env)
        self.unwrapped.wrapped = True
        self.min_cte, self.max_reward, self.min_reward = min_cte, max_reward, min_reward

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        reward += linear_reward(info["cte"], self.min_cte, self.max_reward, self.min_reward)
        return observation, reward, terminated, truncated, info


class _CTELinearVec(_VecWrapper):
    def __init__(self, env, min_cte: float, max_reward: float = 1.0, min_reward: float = 0.0):
        super().__init__(env)
        self.min_cte, self.max_reward, self.min_reward = min_cte, max_reward, min_reward

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        reward = reward + self._live(linear_reward_tensor(info["cte"], self.min_cte, self.max_reward, self.min_reward))
        return observation, reward, terminated, truncated, info


class CTELinearRewardWrapper:
    """reward += linear_reward(cte, min_cte, max_reward, min_reward) (reward.py:64-84)."""
    __new__ = _make(_CTELinearScalar, _CTELinearVec)


# ------------------------------------------------------------------------------------------------ route progress
# An extension (the reference has no navigation task): needs the config's `navigation` section.
class _RouteProgressScalar(Wrapper):
    def __init__(self, env, progress_scale: float = 1.0, goal_bonus: float = 0.0):
        super().__init__(env)
        self.unwrapped.wrapped = True
        self.progress_scale, self.goal_bonus = progress_scale, goal_bonus

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        if "route_progress" not in info:
            raise ValueError("RouteProgressRewardWrapper needs the config's `navigation` section")
        reward += self.progress_scale * info["route_progress"] + self.goal_bonus * float(info["goal_reached"])
        return observation, reward, terminated, truncated, info


class _RouteProgressVec(_VecWrapper):
    def __init__(self, env, progress_scale: float = 1.0, goal_bonus: float = 0.0):
        super().__init__(env)
        if getattr(self.unwrapped, "route", None) is None:
            raise ValueError("RouteProgressRewardWrapper needs the config's `navigation` section")
        self.progress_scale, self.goal_bonus = progress_scale, goal_bonus

    def step(self, action):
        observation, reward, terminated, truncated, info = self.env.step(action)
        term = self.progress_scale * info["route_progress"] + self.goal_bonus * info["goal_reached"].to(torch.float32)
        reward = reward + self._live(term)
        return observation, reward, terminated, truncated, info


class RouteProgressRewardWrapper:
    """reward += progress_scale * route_progress + goal_bonus * goal_reached: metres gained along the route to the goal, and
    a bonus on the step a goal is reached (the config's `navigation` section)."""
    __new__ = _make(_RouteProgressScalar, _RouteProgressVec)


for _pub, _impls in ((LanelineSparseRewardWrapper, (_LanelineSparseScalar, _LanelineSparseVec)),
                     (LanelineLinearRewardWrapper, (_LanelineLinearScalar, _LanelineLinearVec)),
                     (CTESparseRewardWrapper, (_CTESparseScalar, _CTESparseVec)), (CTELinearRewardWrapper, (_CTELinearScalar, _CTELinearVec)),
                     (RouteProgressRewardWrapper, (_RouteProgressScalar, _RouteProgressVec))):
    for _i in _impls:
        _i.__name__ = _pub.__name__
