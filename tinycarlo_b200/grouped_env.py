"""Per-env camera resolution (BASELINE config 5: domain-randomised resolution) by grouping.

A dense [N,C,H,W] tensor cannot hold mixed resolutions, so envs that share a resolution form a group with its own dense
tensors and its own library handle (SURVEY H10). TinyCarloGroupedVecEnv presents the groups as one env: global env
indices (and therefore spawn seeds) run through the groups in order, actions are given for all envs at once, the small
per-env results come back concatenated and the observations as one tensor per group. The groups' kernels are enqueued on
separate CUDA streams so that small groups overlap."""
import copy
from typing import Any, Dict, List, Optional, Sequence, Tuple, Union

import torch

from .config import load_config
from .vec_env import TinyCarloVecEnv


class TinyCarloGroupedVecEnv:
    is_vector_env = True

    def __init__(self, config: Union[str, Dict[str, Any]], groups: Sequence[Tuple[int, Sequence[int]]], device="cuda",
                 env_index_offset: int = 0, group_index_offsets: Optional[Sequence[int]] = None, overlap: bool = True, **kw):
        """groups: [(num_envs, [H, W]), ...]. group_index_offsets: global index of each group's env 0 (default: the groups follow
        each other from env_index_offset on); a multi-GPU job gives every rank a contiguous slice of EVERY group
        (distributed.shard_groups), so that env seeds and per-env parameters do not depend on the sharding. overlap: enqueue
        the groups on separate streams (False: one after the other on the caller's stream). Other arguments as TinyCarloVecEnv."""
        cfg, path = load_config(config)
        self.envs: List[TinyCarloVecEnv] = []
        self.offsets = [0]
        for n, res in groups:
            c = copy.deepcopy(cfg)
            c["camera"]["resolution"] = [int(res[0]), int(res[1])]
            if path is not None and "json_path" in c["map"]:   # keep json_path relative to the yaml's directory
                import os
                c["map"]["json_path"] = os.path.join(os.path.dirname(path), c["map"]["json_path"])
            goff = env_index_offset + self.offsets[-1] if group_index_offsets is None else int(group_index_offsets[len(self.envs)])
            self.envs.append(TinyCarloVecEnv(c, int(n), device=device, env_index_offset=goff, **kw))
            self.offsets.append(self.offsets[-1] + int(n))
        self.num_envs = self.offsets[-1]
        self.device = self.envs[0].device
        self.class_names = self.envs[0].class_names
        self.track_width = self.envs[0].track_width
        self.autoreset = self.envs[0].autoreset
        self.overlap = bool(overlap)
        self._streams = [torch.cuda.Stream(device=self.device) for _ in self.envs]

    @property
    def unwrapped(self):
        return self

    def _slices(self):
        return [slice(a, b) for a, b in zip(self.offsets[:-1], self.offsets[1:])]

    def _fan_out(self, fn):
        """run fn(env, slice) for every group on its own stream, ordered after the caller's stream and joined back"""
        if not self.overlap:
            return [fn(env, sl) for env, sl in zip(self.envs, self._slices())]
        cur = torch.cuda.current_stream(self.device)
        start = torch.cuda.Event()
        start.record(cur)
        outs = []
        for env, sl, st in zip(self.envs, self._slices(), self._streams):
            st.wait_event(start)
            with torch.cuda.stream(st):
                outs.append(fn(env, sl))
            done = torch.cuda.Event()
            done.record(st)
            cur.wait_event(done)
        return outs

    @staticmethod
    def _cat_info(infos):
        return {k: torch.cat([i[k] for i in infos], dim=0) for k in infos[0]}

    def set_wrapped(self, wrapped: bool = True):
        for e in self.envs:
            e.set_wrapped(wrapped)

    def mark_done(self, mask: torch.Tensor):
        for e, sl in zip(self.envs, self._slices()):
            e.mark_done(mask[sl])

    def reset(self, seed: Optional[int] = None, mask: Optional[torch.Tensor] = None):
        outs = self._fan_out(lambda e, sl: e.reset(seed=seed, mask=None if mask is None else mask[sl]))
        return [o[0] for o in outs], self._cat_info([o[1] for o in outs])

    def step(self, action: Dict[str, torch.Tensor]):
        cc, man = action["car_control"], action["maneuver"]
        outs = self._fan_out(lambda e, sl: e.step({"car_control": cc[sl], "maneuver": man[sl]}))
        return ([o[0] for o in outs], torch.cat([o[1] for o in outs]), torch.cat([o[2] for o in outs]), torch.cat([o[3] for o in outs]),
                self._cat_info([o[4] for o in outs]))

    def reset_done(self):
        outs = self._fan_out(lambda e, sl: e.reset_done())
        return [o[0] for o in outs], self._cat_info([o[1] for o in outs])

    def set_camera_params(self, env_ids=None, camera=None, **kw):
        """per-env camera parameters by GLOBAL env index (arrays cover all envs when env_ids is None); camera: the rig's
        camera index or indices, as TinyCarloVecEnv.set_camera_params (the config's `cameras` list applies to every group)"""
        import numpy as np
        ids = np.arange(self.num_envs) if env_ids is None else np.asarray(env_ids).reshape(-1)
        for e, (a, b) in zip(self.envs, zip(self.offsets[:-1], self.offsets[1:])):
            sel = (ids >= a) & (ids < b)
            if not sel.any():
                continue
            sub = {}
            for k, v in kw.items():
                if v is None:
                    continue
                v = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
                sub[k] = v[sel] if v.ndim >= 1 and len(v) == len(ids) else v
            e.set_camera_params(env_ids=ids[sel] - a, camera=camera, **sub)

    def set_car_params(self, **kw):
        import numpy as np
        for e, (a, b) in zip(self.envs, zip(self.offsets[:-1], self.offsets[1:])):
            sub = {}
            for k, v in kw.items():
                if v is None or np.ndim(v) == 0:
                    sub[k] = v
                else:
                    v = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
                    sub[k] = v[a:b]
            e.set_car_params(**sub)

    @property
    def launch_count(self) -> int:
        return sum(e.launch_count for e in self.envs)

    @property
    def reset_mask(self) -> torch.Tensor:
        return torch.cat([e.reset_mask for e in self.envs])

    @property
    def obs_bytes_per_step(self) -> int:
        return sum(e.obs.numel() * e.obs.element_size() for e in self.envs)

    def close(self):
        for e in self.envs:
            e.close()
