"""The reference's wrappers (tinycarlo/wrapper/__init__.py:1-3) for the single-env drop-in and the vectorised env.
NoiseObservationWrapper is provided with a defined (seeded, counter-based) RNG contract: the reference draws from the unseeded
global np.random, so its noise cannot be reproduced, only its operation (wrapper/observation.py here)."""
from .reward import (CTELinearRewardWrapper, CTESparseRewardWrapper, LanelineLinearRewardWrapper, LanelineSparseRewardWrapper,  # noqa: F401
                     RouteProgressRewardWrapper)
from .termination import CrashTerminationWrapper, CTETerminationWrapper, LanelineCrossingTerminationWrapper  # noqa: F401
from .utils import linear_reward, sparse_reward  # noqa: F401


def __getattr__(name):   # lazy: the noise wrapper needs torch + the CUDA library
    if name == "NoiseObservationWrapper":
        from .observation import NoiseObservationWrapper
        return NoiseObservationWrapper
    raise AttributeError(name)
