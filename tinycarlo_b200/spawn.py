"""Spawn-node draws with the reference's RNG semantics (tinycarlo/map.py:51-69 under gymnasium seeding).

gymnasium's Env.reset(seed=s) installs np.random.Generator(PCG64(SeedSequence(s))); each reset then makes one bounded
draw (choice(spawn_points), or integers(0, n_nodes-1) without spawn points) and redraws while the node has no
successor. Env i of a vectorised env is seeded with seed + global_index(i), like gymnasium.vector.

The product draws on the DEVICE: spawn_stream_states() seeds one PCG64 stream per env on the host (SeedSequence hashing,
tinycarlo_b200/pcg64.py) and the reset paths of the tracking kernel advance it (tc_spawn_draw in csrc/tc_core.cuh), so
resets never synchronise with the host. SpawnSampler is the host model of the same streams on numpy arrays: it tells
what the device must draw (tests, tools) and is not on the step path."""
from typing import Optional

import numpy as np

from .maptables import MapTables
from .pcg64 import VecPCG64


def make_generator(seed: Optional[int]) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed)))


def stream_seeds(num_envs: int, seed: Optional[int], env_index_offset: int = 0) -> np.ndarray:
    if seed is None:   # OS entropy, one independent stream per env
        return np.random.SeedSequence().generate_state(int(num_envs), np.uint64)
    return np.arange(int(num_envs), dtype=np.uint64) + np.uint64(int(seed) + int(env_index_offset))


def spawn_stream_states(num_envs: int, seed: Optional[int], env_index_offset: int = 0) -> np.ndarray:
    """uint64 [num_envs, 5] in the layout of include/tinycarlo_b200.h TC_RNG_*: the freshly seeded
    Generator(PCG64(SeedSequence(seed + offset + i))) of every env (state hi, lo, increment hi, lo, empty 32-bit buffer)."""
    return VecPCG64(stream_seeds(num_envs, seed, env_index_offset)).device_rows()


def goal_stream_states(num_envs: int, seed: Optional[int], env_index_offset: int = 0, seeds: Optional[np.ndarray] = None) -> np.ndarray:
    """The goal streams of the navigation goals (include/tinycarlo_b200.h TcRouteDesc) in the same row layout: env i gets
    Generator(PCG64(SeedSequence(seed + offset + i).spawn(1)[0])), the first child of its spawn stream's seed sequence, so the
    spawn draws stay what they are without goals. seeds: the per-env seeds stream_seeds() returned for the spawn streams (with
    seed None, the same OS entropy)."""
    if seeds is None:
        seeds = stream_seeds(num_envs, seed, env_index_offset)
    return VecPCG64(seeds, spawn_key=(0,)).device_rows()


class SpawnSampler:
    def __init__(self, tables: MapTables, num_envs: int, table_len: int = 16, env_index_offset: int = 0):
        self.tables, self.n, self.K, self.offset = tables, int(num_envs), int(table_len), int(env_index_offset)
        self.rng: Optional[VecPCG64] = None
        self.table = None  # int32 [n, K]: the next K spawn nodes of every env
        sp = tables.spawn_points
        self._choices = None if sp is None else np.asarray(sp, np.int64)

    def _draw(self, m: np.ndarray) -> np.ndarray:
        """one spawn node for every env selected by the boolean mask m (map.py:61-64, redraw while no successor)"""
        out = np.zeros(self.n, np.int64)
        pending = m.copy()
        t = self.tables
        while pending.any():
            if self._choices is None:
                idx = self.rng.bounded(len(t.lp_nodes) - 1, pending)      # integers(0, len(nodes)-1): never the last node
            else:
                idx = self._choices[self.rng.bounded(len(self._choices), pending)]   # choice(spawn_points)
            where = np.nonzero(pending)[0]
            ok = t.has_successor[idx]
            out[where[ok]] = idx[ok]
            pending[where[ok]] = False
        return out[m]

    def seed(self, seed: Optional[int]):
        self.rng = VecPCG64(stream_seeds(self.n, seed, self.offset))
        tab = np.empty((self.n, self.K), np.int32)
        all_envs = np.ones(self.n, bool)
        for k in range(self.K):
            tab[:, k] = self._draw(all_envs)
        self.table = tab
        return tab

    def advance(self, consumed: np.ndarray):
        """Env i used its first consumed[i] entries: shift them out and draw as many new ones at the end."""
        K = self.K
        c = np.minimum(np.asarray(consumed, np.int64), K)
        if not c.any():
            return self.table
        tab = self.table
        src = np.arange(K)[None, :] + c[:, None]                   # column j takes old column j + c_i when that exists
        new = np.where(src < K, np.take_along_axis(tab, np.minimum(src, K - 1), axis=1), -1).astype(np.int32)
        for r in range(int(c.max())):                               # r-th fresh draw of every env that needs one
            m = c > r
            new[m, K - c[m] + r] = self._draw(m)
        self.table = new
        return new

    def state_dict(self):
        return {"table": self.table.copy(), "rng": self.rng.state_dict()}

    def load_state_dict(self, d):
        self.table = np.array(d["table"], np.int32)
        self.rng = VecPCG64()
        self.rng.load_state_dict(d["rng"])
