"""TinyCarloVecEnv — N tinycarlo environments stepped in lockstep on one B200, CUDA tensors in and out.

The vectorised counterpart of the reference's TinyCarloEnv (tinycarlo/env.py:15-147): same config schema, same action
dict ({"car_control": [velocity cmd, steering cmd] in [-1,1], "maneuver": 0..3}), same observation formats and the
same info keys, batched along dim 0. One step() enqueues two hand-written sm_100a kernels through the C ABI (tracking;
fused camera pass + rasterise + store) on torch's current stream and returns views of preallocated tensors; there is no
host synchronisation inside step() - resets and spawn draws included, so a rollout loop can be captured in a CUDA graph -
and no CPU implementation.

Returned tensors are owned by the env and are overwritten by the next step()/reset(); clone what must survive.
"""
import ctypes as C
import os
from typing import Any, Callable, Dict, Optional, Union

import numpy as np
import torch

from . import _lib
from .camera_params import camera_row
from .config import LINE_THICKNESS_MAX, bev_params, camera_params, car_param_row, load_config, resolve_map_path, sim_params
from .maptables import MapTables
from .spawn import spawn_stream_states


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class TinyCarloVecEnv:
    is_vector_env = True

    def __init__(self, config: Union[str, Dict[str, Any]], num_envs: int, device: Union[str, int, torch.device] = "cuda",
                 obs_format: Optional[str] = None, env_index_offset: int = 0, debug_segments: bool = False,
                 autoreset: Optional[str] = None):
        """config: yaml path / directory / dict as for the reference env. num_envs: envs on THIS device.
        env_index_offset: global index of local env 0 (multi-GPU sharding: env i is seeded with seed + offset + i, so
        results do not depend on how the envs are sharded). debug_segments: also export the projected int32 segments.
        autoreset: None (the reference's behaviour: the caller resets finished envs, see reset(mask=...) / reset_done()) or
        "next_step" (gymnasium's AutoresetMode.NEXT_STEP, done inside the step kernel with no extra launch: the step after an
        env terminated or truncated resets it, ignores its action and returns the reset observation with reward 0)."""
        if not torch.cuda.is_available():
            raise _lib.TinyCarloError("TinyCarloVecEnv needs a CUDA device: there is no CPU implementation")
        self.config, self.config_path = load_config(config)
        sp = sim_params(self.config)
        self.fps, self.T = sp["fps"], sp["T"]
        self.observation_space_format = obs_format or sp["observation_space_format"]
        self.map = MapTables(resolve_map_path(self.config["map"], self.config_path), self.config["map"]["pixel_per_meter"],
                             self.config["map"].get("spawn_points", None))
        self.cam_cfg = camera_params(self.config["camera"])
        self.num_envs = int(num_envs)
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.env_index_offset = int(env_index_offset)
        self.H, self.W = (int(v) for v in self.cam_cfg["resolution"])
        self.n_classes = self.map.n_classes
        self.class_names = self.map.get_laneline_names()
        self.track_width = float(self.config["car"].get("track_width", 0.03))
        self.wrapped = False
        self.no_observation = False
        N, Cn = self.num_envs, self.n_classes
        dev = self.device
        fmt = {"rgb": _lib.TC_OBS_RGB, "classes_bits": _lib.TC_OBS_CLASSES_BITS, "classes_bf16": _lib.TC_OBS_CLASSES_BF16}.get(
            self.observation_space_format, _lib.TC_OBS_CLASSES)
        self._fmt = fmt
        # "classes" (u8 0/255, the reference's format), "rgb", and two formats a policy can consume directly:
        # "classes_bits": int32 [N,C,ceil(H*W/32)], bit (y*W+x)%32 of word (y*W+x)/32 is pixel (x,y)  (8x fewer bytes)
        # "classes_bf16": bfloat16 [N,C,H,W] with 0.0 / 1.0
        self.obs_shape = {_lib.TC_OBS_CLASSES: (Cn, self.H, self.W), _lib.TC_OBS_RGB: (self.H, self.W, 3),
                          _lib.TC_OBS_CLASSES_BITS: (Cn, (self.H * self.W + 31) // 32), _lib.TC_OBS_CLASSES_BF16: (Cn, self.H, self.W)}[fmt]
        self.obs_dtype = {_lib.TC_OBS_CLASSES_BITS: torch.int32, _lib.TC_OBS_CLASSES_BF16: torch.bfloat16}.get(fmt, torch.uint8)

        # ---- library handle (map tables go to the device once)
        m = self.map
        self._keep = [np.ascontiguousarray(a) for a in (m.ll_node_off, m.ll_edge_off, m.ll_nodes, m.ll_edges, m.colors, m.lp_nodes,
                                                        m.lp_edges, m.lp_orient, m.lp_orient_rev)]
        k = self._keep
        desc = _lib.TcMapDesc(Cn, k[0].ctypes.data, k[1].ctypes.data, k[2].ctypes.data, k[3].ctypes.data, k[4].ctypes.data,
                              len(m.lp_nodes), len(m.lp_edges), k[5].ctypes.data, k[6].ctypes.data, k[7].ctypes.data, k[8].ctypes.data)
        sim = _lib.TcSimDesc(self.H, self.W, fmt)
        self._L = _lib.lib()
        h = C.c_void_p()
        _lib.check(self._L.tc_create(C.byref(desc), C.byref(sim), N, self.device.index, C.byref(h)), "tc_create")
        self._h = h

        # ---- outputs (allocated once; step()/reset() return views)
        with torch.cuda.device(dev):
            self.obs = torch.zeros((N,) + self.obs_shape, dtype=self.obs_dtype, device=dev)
            f32 = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)  # noqa: E731
            self.out = {"cte": f32(N), "heading_error": f32(N), "velocity": f32(N), "reward": f32(N), "position": f32(N, 2),
                        "orientation": f32(N), "laneline_distances": f32(N, Cn),
                        "nearest_edge": torch.full((N, Cn), -1, dtype=torch.int32, device=dev), "local_path": f32(N, 4, 2),
                        "local_path_nodes": torch.full((N, 4, 2), -1, dtype=torch.int32, device=dev),
                        "path_len": torch.zeros(N, dtype=torch.int32, device=dev),
                        "terminated": torch.zeros(N, dtype=torch.uint8, device=dev),
                        "truncated": torch.zeros(N, dtype=torch.uint8, device=dev),
                        "info_f64": torch.zeros((N, 4 + Cn), dtype=torch.float64, device=dev)}
            if debug_segments:
                self.out["seg_count"] = torch.zeros((N, Cn), dtype=torch.int32, device=dev)
                self.out["seg_i32"] = torch.zeros((N, max(int(m.ll_edge_off[-1]), 1), 4), dtype=torch.int32, device=dev)
            # bird's-eye view (config section `bev`, tc_set_bev): [N,P,H,W] u8 or [N,P,H*W/32] int32, rewritten by every
            # step() / reset() whatever no_observation says; None without the section
            self.bev_cfg = bev_params(self.config, Cn)
            self.bev = None
            if self.bev_cfg is not None:
                b = self.bev_cfg
                bh, bw = b["resolution"]
                bits = b["format"] == "classes_bits"
                self.bev = torch.zeros((N, b["planes"]) + ((bh * bw // 32,) if bits else (bh, bw)), dtype=torch.int32 if bits else torch.uint8,
                                       device=dev)
                bdesc = _lib.TcBevDesc(bh, bw, b["pixel_per_meter"], b["car_pixel"][0], b["car_pixel"][1], b["line_thickness"], int(b["route"]),
                                       _lib.TC_OBS_CLASSES_BITS if bits else _lib.TC_OBS_CLASSES)
                _lib.check(self._L.tc_set_bev(self._h, C.byref(bdesc), _ptr(self.bev)), "tc_set_bev")
            self._spawn_nodes = torch.full((N,), -1, dtype=torch.int32, device=dev)   # node of each env's latest reset
            self._mask_all = torch.ones(N, dtype=torch.uint8, device=dev)
        self._outs = self._make_outputs(with_obs=True)
        self._outs_noobs = self._make_outputs(with_obs=False)

        # ---- parameters
        self._car_rows = np.tile(np.array(car_param_row(self.config["car"], self.T), np.float64), (N, 1))
        cc = self.cam_cfg
        self._cam_rows = np.tile(camera_row(cc["position"], cc["orientation"], cc["fov"], cc["resolution"], cc["max_range"]), (N, 1))
        self._thickness = np.full(N, int(cc["line_thickness"]), np.int32)
        self._check_car_rows(self._car_rows)
        self._upload_params()

        # ---- spawn draws (map.py:51-69) on the device: one numpy-compatible PCG64 stream per env, seeded like gymnasium
        # (Generator(PCG64(SeedSequence(seed + global index)))) on the host and advanced inside the reset paths of the
        # tracking kernel, so resets and autoresets never synchronise with the host.
        if autoreset not in (None, "next_step"):
            raise ValueError("autoreset must be None or 'next_step'")
        self.autoreset = autoreset
        with torch.cuda.device(dev):
            self._rng_state = torch.zeros((N, _lib.TC_RNG_N), dtype=torch.int64, device=dev)   # uint64 bit patterns
            sp = self.map.spawn_points
            self._spawn_points = None if sp is None else torch.tensor(sp, dtype=torch.int32, device=dev)
            self.done_flags = torch.zeros(N, dtype=torch.uint8, device=dev) if autoreset else None
            # autoreset: which envs the latest step() reset instead of advancing (all zero otherwise)
            self._reset_mask = torch.zeros(N, dtype=torch.uint8, device=dev)
        _lib.check(self._L.tc_set_spawn_rng(self._h, _ptr(self._rng_state), _ptr(self._spawn_points), 0 if sp is None else len(sp),
                                            _ptr(self._spawn_nodes)), "tc_set_spawn_rng")
        if autoreset:
            _lib.check(self._L.tc_set_autoreset(self._h, _ptr(self.done_flags)), "tc_set_autoreset")
            _lib.check(self._L.tc_set_reset_mask(self._h, _ptr(self._reset_mask)), "tc_set_reset_mask")
        self._seeded = False
        self._was_reset = False   # step() before the first reset() raises (the reference resets in its constructor)
        # tinycarlo/helper.py:4 getenv("DEBUG"): per-phase milliseconds printed after every step (env.py:144-145); here the
        # phases are the two kernels, timed with CUDA events - this mode synchronises, the normal one never does
        self._debug = os.environ.get("DEBUG", "").lower() == "1"

    # ------------------------------------------------------------------------------------------------ plumbing
    def _make_outputs(self, with_obs: bool) -> _lib.TcOutputs:
        o = _lib.TcOutputs()
        for name in _lib.OUTPUT_FIELDS:
            t = self.obs if name == "obs" else self.out.get(name)
            if name == "obs" and not with_obs:
                t = None
            setattr(o, name, None if t is None else t.data_ptr())
        # what step() hands back is the same set of tensors every time: build the views and the info dict once (a step is two
        # kernel launches; at a few thousand small frames the Python around them shows in the eager env-steps/s)
        self._flag_views = (self.out["terminated"].view(torch.bool), self.out["truncated"].view(torch.bool))
        self._info_cache = self._info()
        return o

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _upload_params(self):
        """Car and camera rows to the device. Nothing here waits for the device: the library decides from the host copy of the
        camera rows which visible-set tables to use (tc_set_camera_params_host) and keeps the tables it has built."""
        with torch.cuda.device(self.device):
            car = torch.from_numpy(self._car_rows).to(self.device)
            cam = torch.from_numpy(self._cam_rows).to(self.device)
            th = torch.from_numpy(self._thickness).to(self.device)
            rows = np.ascontiguousarray(self._cam_rows, np.float64)
            _lib.check(self._L.tc_set_car_params(self._h, _ptr(car), self._stream()), "tc_set_car_params")
            _lib.check(self._L.tc_set_camera_params_host(self._h, _ptr(cam), _ptr(th), C.c_void_p(rows.ctypes.data), self._stream()),
                       "tc_set_camera_params")
            self._param_staging = (car, cam, th)   # alive until the next upload: the copies above are stream-ordered

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.tc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------ parameters
    def set_wrapped(self, wrapped: bool = True):
        """env.py:137-138: wrappers switch the default reward/termination off."""
        self.wrapped = bool(wrapped)
        _lib.check(self._L.tc_set_wrapped(self._h, int(self.wrapped)), "tc_set_wrapped")

    def set_car_params(self, **kw):
        """Per-env car parameters (domain randomisation). Each value: scalar or array [N]; None = unlimited where the
        reference allows it (steering_speed, max_acceleration). Keys as in the config's `car` section."""
        cols = {"wheelbase": 0, "track_width": 1, "max_velocity": 2, "max_steering_angle": 3, "steering_speed": 4,
                "max_acceleration": 5, "max_deceleration": 6}
        rows = self._car_rows.copy()
        for key, val in kw.items():
            col = cols[key]
            if val is None:
                if key not in ("steering_speed", "max_acceleration"):
                    raise ValueError(f"car.{key} cannot be None")
                rows[:, col] = np.nan
            else:
                v = val.detach().cpu().numpy() if isinstance(val, torch.Tensor) else np.asarray(val, np.float64)
                rows[:, col] = v
        self._check_car_rows(rows)
        self._car_rows = rows
        self._upload_params()

    @staticmethod
    def _check_car_rows(rows: np.ndarray):
        """Rejects parameters that make the bicycle model degenerate (wheelbase 0 divides by zero in car.py:103, a non-finite
        value poisons every env that reads it); the reference accepts them and produces inf / NaN poses."""
        for col, name, positive in ((0, "wheelbase", True), (1, "track_width", True), (2, "max_velocity", False),
                                    (3, "max_steering_angle", False), (6, "max_deceleration", False), (7, "dt", True)):
            v = rows[:, col]
            if name == "max_deceleration":
                v = v[~np.isnan(rows[:, 5])]   # only read when max_acceleration is set (car.py:81-82)
            if not np.all(np.isfinite(v)) or (positive and not np.all(v > 0)):
                raise ValueError(f"car.{name} must be finite" + (" and > 0" if positive else ""))

    @staticmethod
    def _thickness_rows(v, shape) -> np.ndarray:
        """Per-env line thicknesses as int32 of `shape`: integers in 1..255 like the config's camera.line_thickness (0 and
        negative values would draw 1-pixel lines where cv2.polylines raises; larger ones leave the rasteriser's 16.16 range)."""
        a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        if a.dtype == np.bool_ or not np.issubdtype(a.dtype, np.integer) or not ((a >= 1) & (a <= LINE_THICKNESS_MAX)).all():
            raise ValueError(f"camera.line_thickness must be integers in 1..{LINE_THICKNESS_MAX}, got {v!r}")
        return np.broadcast_to(a, shape).astype(np.int32)

    def set_camera_params(self, position=None, orientation=None, fov=None, max_range=None, line_thickness=None, env_ids=None):
        """Per-env camera parameters (camera.py:48-50 update_params, vectorised). Arrays are [n,3] / [n] for the envs in
        env_ids (default: all), or a single value broadcast. E and K are rebuilt on the host with the reference's calls."""
        ids = np.arange(self.num_envs) if env_ids is None else np.asarray(env_ids).reshape(-1)
        n = len(ids)
        thickness = None if line_thickness is None else self._thickness_rows(line_thickness, (n,))
        if not hasattr(self, "_cam_src"):
            cc = self.cam_cfg
            self._cam_src = {"position": np.tile(np.asarray(cc["position"], np.float64), (self.num_envs, 1)),
                             "orientation": np.tile(np.asarray(cc["orientation"], np.float64), (self.num_envs, 1)),
                             "fov": np.full(self.num_envs, float(cc["fov"])), "max_range": np.full(self.num_envs, float(cc["max_range"]))}

        def bc(v, shape):
            v = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v, np.float64)
            return np.broadcast_to(v, shape)
        if position is not None:
            self._cam_src["position"][ids] = bc(position, (n, 3))
        if orientation is not None:
            self._cam_src["orientation"][ids] = bc(orientation, (n, 3))
        if fov is not None:
            self._cam_src["fov"][ids] = bc(fov, (n,))
        if max_range is not None:
            self._cam_src["max_range"][ids] = bc(max_range, (n,))
        if thickness is not None:
            self._thickness[ids] = thickness
        res = [self.H, self.W]
        s = self._cam_src
        cache = {}
        for i in ids:
            key = (tuple(s["position"][i]), tuple(s["orientation"][i]), float(s["fov"][i]), float(s["max_range"][i]))
            row = cache.get(key)
            if row is None:
                row = cache[key] = camera_row(s["position"][i], s["orientation"][i], s["fov"][i], res, s["max_range"][i])
            self._cam_rows[i] = row
        self._upload_params()

    def set_camera_rows(self, cam_rows: np.ndarray, line_thickness=None):
        """Raw per-env camera rows [N,20] (E 3x4 row-major, fx, fy, cx, cy, max_range, pad) — include/tinycarlo_b200.h TC_CAM_*."""
        thickness = None if line_thickness is None else self._thickness_rows(line_thickness, (self.num_envs,))
        self._cam_rows[:] = np.asarray(cam_rows, np.float64).reshape(self.num_envs, _lib.TC_CAM_N)
        if thickness is not None:
            self._thickness[:] = thickness
        self._upload_params()

    # ------------------------------------------------------------------------------------------------ spawn draws
    def _seed(self, seed: Optional[int]):
        st = spawn_stream_states(self.num_envs, seed, self.env_index_offset)
        with torch.cuda.device(self.device):
            self._rng_state.copy_(torch.from_numpy(st.view(np.int64)))   # in place: the library holds the address
        self._seeded = True

    # ------------------------------------------------------------------------------------------------ gym-like API
    def _info(self) -> Dict[str, torch.Tensor]:
        o = self.out
        info = {"cte": o["cte"], "heading_error": o["heading_error"], "position": o["position"], "orientation": o["orientation"],
                "laneline_distances": o["laneline_distances"], "local_path": o["local_path"], "velocity": o["velocity"],
                "nearest_edge": o["nearest_edge"], "local_path_nodes": o["local_path_nodes"], "path_len": o["path_len"]}
        if self.bev is not None:
            info["bev"] = self.bev
        return info

    def reset(self, seed: Optional[int] = None, mask: Optional[torch.Tensor] = None, spawn_nodes: Optional[torch.Tensor] = None):
        """env.py:101-113 for the envs selected by `mask` (bool/uint8 [N]; None = all). seed re-seeds every env's spawn
        generator (env i gets seed + env_index_offset + i, as gymnasium.vector does). spawn_nodes (int32 [N]) overrides
        the draw (tests). Returns (obs, info); info of reset envs is the reference's empty info (zeros)."""
        with torch.cuda.device(self.device):
            if seed is not None or not self._seeded:
                self._seed(seed)
            if mask is not None:
                mask_u8 = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            else:
                mask_u8 = self._mask_all
            nodes = None   # NULL: every selected env draws from its own device stream
            if spawn_nodes is not None:
                nodes = spawn_nodes.to(device=self.device, dtype=torch.int32).contiguous()
            if self.autoreset:
                self.done_flags.masked_fill_(mask_u8.bool(), 0)
            outs = self._outs if not self.no_observation else self._outs_noobs
            _lib.check(self._L.tc_reset(self._h, _ptr(mask_u8), _ptr(nodes), C.byref(outs), self._stream()), "tc_reset")
            self._was_reset = True
        return self.obs, self._info()

    def step(self, action: Dict[str, torch.Tensor]):
        """env.py:115-147 for all envs. action["car_control"]: float [N,2] (velocity cmd, steering cmd), action["maneuver"]:
        int [N]. Returns (obs, reward f32[N], terminated bool[N], truncated bool[N], info dict of tensors)."""
        cc = action["car_control"]
        man = action["maneuver"]
        if cc.dtype not in (torch.float32, torch.float64):
            cc = cc.to(torch.float32)
        cc = cc.contiguous()              # keeps the dtype: a float64 slice stays on the float64 entry point
        f64 = cc.dtype == torch.float64   # float64 actions keep the reference's float64 path bit for bit
        if man.dtype != torch.int32 or not man.is_contiguous():
            man = man.to(torch.int32).contiguous()
        if cc.device != self.device or man.device != self.device or cc.shape != (self.num_envs, 2) or man.shape != (self.num_envs,):
            raise ValueError("action tensors must live on the env's device with shapes [N,2] and [N]")
        outs = self._outs if not self.no_observation else self._outs_noobs
        if not self._was_reset:
            raise _lib.TinyCarloError("call reset() before step()")
        fn = self._L.tc_step_f64 if f64 else self._L.tc_step
        if self._debug and not torch.cuda.is_current_stream_capturing():
            with torch.cuda.device(self.device):
                self.profile_begin(1)
                _lib.check(fn(self._h, _ptr(cc), _ptr(man), C.byref(outs), self._stream()), "tc_step")
                ms, _ = self.profile_end()
            print(f"all: {ms['track'] + ms['project'] + ms['raster']:.3f} ms | obs render {ms['project'] + ms['raster']:.3f} ms | "
                  f"car step + info {ms['track']:.3f} ms  ({self.num_envs} envs)")
        elif torch.cuda.current_device() == self.device.index:   # the usual case: skip the device context manager (~10 us of Python)
            _lib.check(fn(self._h, _ptr(cc), _ptr(man), C.byref(outs), self._stream()), "tc_step")
        else:
            with torch.cuda.device(self.device):
                _lib.check(fn(self._h, _ptr(cc), _ptr(man), C.byref(outs), self._stream()), "tc_step")
        return self.obs, self.out["reward"], self._flag_views[0], self._flag_views[1], dict(self._info_cache)

    def capture(self, policy_fn: Optional[Callable[["TinyCarloVecEnv"], Dict[str, torch.Tensor]]] = None, steps: int = 1,
                warmup: int = 3) -> "torch.cuda.CUDAGraph":
        """Captures `steps` iterations of `action = policy_fn(env); env.step(action)` in a CUDA graph and returns it; every
        graph.replay() then advances all envs by `steps` steps with a single launch (step() neither allocates nor synchronises,
        and resets happen inside the kernels with autoreset="next_step"). policy_fn must only enqueue work on the current
        stream and write into tensors it owns; results are read from env.obs / env.out afterwards. The launch-bound small
        configurations (BASELINE config 2: 4096 envs at 84x84) gain the most. The warm-up steps and the captured call itself
        do advance / not advance the envs respectively, as torch's capture rules imply."""
        if self.autoreset is None and steps > 1:
            raise ValueError("capturing several steps needs autoreset='next_step' (nothing else resets finished envs inside a graph)")
        if not self._was_reset:
            raise _lib.TinyCarloError("call reset() before capture()")
        dbg, self._debug = self._debug, False

        def one():
            if policy_fn is None:
                raise ValueError("capture() needs a policy_fn(env) -> action dict")
            self.step(policy_fn(self))
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(max(int(warmup), 1)):
                one()
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(int(steps)):
                one()
        self._debug = dbg
        return graph

    def reset_done(self):
        """Resets the envs whose last step terminated or truncated, as a caller of the reference would (on the device, no
        host sync). With autoreset="next_step" this is unnecessary: the next step() does it inside the kernel."""
        done = self.out["terminated"] | self.out["truncated"]
        return self.reset(mask=done)

    @property
    def reset_mask(self) -> torch.Tensor:
        """bool [N]: the envs that the latest step() reset instead of advancing (autoreset="next_step"); their reward is 0,
        their info empty and their observation the spawn frame. All False without autoreset."""
        return self._reset_mask.view(torch.bool)

    def mark_done(self, mask: torch.Tensor):
        """autoreset only: ORs extra termination conditions (e.g. from wrappers) into the flags the next step() consumes."""
        self.done_flags |= mask.to(device=self.device, dtype=torch.uint8)

    def step_host(self, car_control: torch.Tensor, maneuver: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor,
                  truncated: torch.Tensor, cte: Optional[torch.Tensor] = None, heading_error: Optional[torch.Tensor] = None,
                  obs_host: Optional[torch.Tensor] = None):
        """The same step with HOST tensors (ideally pinned): actions are copied to the device, the scalar results copied
        back, and the stream synchronised inside the call (tc_step_host). Observations stay on the device in self.obs unless
        obs_host (a host tensor of self.obs's shape and dtype) is given: then all frames follow in one device-to-host copy
        (tc_step_host_obs; use obs_format="classes_bits" to move an eighth of the bytes)."""
        if not self._was_reset:
            raise _lib.TinyCarloError("call reset() before step_host()")
        for name, t, shape, dt in (("car_control", car_control, (self.num_envs, 2), torch.float32), ("maneuver", maneuver, (self.num_envs,), torch.int32)):
            if t.is_cuda or t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous():
                raise ValueError(f"step_host: {name} must be a contiguous host tensor of dtype {dt} and shape {shape}")
        outs = self._outs if not self.no_observation else self._outs_noobs
        with torch.cuda.device(self.device):
            if obs_host is None:
                _lib.check(self._L.tc_step_host(self._h, _ptr(car_control), _ptr(maneuver), C.byref(outs), _ptr(reward), _ptr(terminated),
                                                _ptr(truncated), _ptr(cte), _ptr(heading_error), self._stream()), "tc_step_host")
            else:
                if obs_host.is_cuda or obs_host.dtype != self.obs.dtype or obs_host.shape != self.obs.shape or not obs_host.is_contiguous():
                    raise ValueError("step_host: obs_host must be a contiguous host tensor with the shape and dtype of env.obs")
                if self.no_observation:
                    raise ValueError("step_host: obs_host given but no_observation is set")
                nbytes = self.obs.numel() * self.obs.element_size()
                _lib.check(self._L.tc_step_host_obs(self._h, _ptr(car_control), _ptr(maneuver), C.byref(outs), _ptr(reward), _ptr(terminated),
                                                    _ptr(truncated), _ptr(cte), _ptr(heading_error), _ptr(obs_host), nbytes, self._stream()),
                           "tc_step_host_obs")

    def render_rgb(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """RGB camera frames [N,H,W,3] at the current poses (renderer.py:36-44), independent of the obs format."""
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.empty((self.num_envs, self.H, self.W, 3), dtype=torch.uint8, device=self.device)
            _lib.check(self._L.tc_render(self._h, None, _ptr(out), _lib.TC_OBS_RGB, None, None, self._stream()), "tc_render")
        return out

    def render_overview(self, env_index: int = 0, overview_pixel_per_meter: Optional[int] = None) -> np.ndarray:
        """Bird's-eye view of the map with env `env_index`'s car and tracked path (renderer.py:19-34): a host-side debugging
        view (reads that env's state back), RGB uint8."""
        from .overview import OverviewRenderer
        ppm = int(overview_pixel_per_meter or self.config["sim"].get("overview_pixel_per_meter", 150))
        if getattr(self, "_overview", None) is None or self._overview.ppm != ppm:
            self._overview = OverviewRenderer(self.map, ppm, node_names=self.config["sim"].get("render_node_names", False))
        st = self.state_dict()
        sf, si = st["sf"][env_index].cpu().numpy(), st["si"][env_index].cpu().numpy()
        path = [(int(si[2 + 2 * i]), int(si[3 + 2 * i])) for i in range(max(int(si[0]), 0))]
        return self._overview.render([float(sf[0]), float(sf[1])], float(sf[2]), float(sf[3]), float(self._car_rows[env_index, 0]),
                                     float(self._car_rows[env_index, 1]), path)

    def render_bev(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Re-render self.bev (the config's `bev` section) at the current poses for the envs in `mask` (None = all)."""
        if self.bev is None:
            raise ValueError("render_bev: the config has no `bev` section")
        with torch.cuda.device(self.device):
            m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
            _lib.check(self._L.tc_render_bev(self._h, _ptr(m), self._stream()), "tc_render_bev")
        return self.bev

    def render_obs(self, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Re-render self.obs at the current poses (after load_state_dict / set_camera_params)."""
        with torch.cuda.device(self.device):
            m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
            _lib.check(self._L.tc_render(self._h, _ptr(m), _ptr(self.obs), self._fmt, _ptr(self.out.get("seg_count")),
                                         _ptr(self.out.get("seg_i32")), self._stream()), "tc_render")
        return self.obs

    # ------------------------------------------------------------------------------------------------ state
    def state_dict(self) -> Dict[str, torch.Tensor]:
        """Car state: sf f64 [N,8] (x, y, rot, steering deg, velocity, front x, front y, pad), si i32 [N,16] (path_len,
        last_maneuver, 4 node pairs, 4 edge ids)."""
        with torch.cuda.device(self.device):
            sf = torch.empty((self.num_envs, _lib.TC_SF_N), dtype=torch.float64, device=self.device)
            si = torch.empty((self.num_envs, _lib.TC_SI_N), dtype=torch.int32, device=self.device)
            _lib.check(self._L.tc_get_state(self._h, _ptr(sf), _ptr(si), self._stream()), "tc_get_state")
        return {"sf": sf, "si": si}

    def checkpoint(self) -> Dict[str, Any]:
        """Everything needed to resume a rollout bit for bit: car state, the spawn streams (per-env PCG64 states) and the
        autoreset flags. The reference has no counterpart (SURVEY section 5)."""
        ck = {k: v.cpu() for k, v in self.state_dict().items()}
        if self._seeded:
            ck["spawn_rng"] = self._rng_state.cpu()
            ck["last_spawn"] = self._spawn_nodes.cpu()
        if self.autoreset:
            ck["done_flags"] = self.done_flags.cpu()
        return ck

    def restore(self, ck: Dict[str, Any]):
        self.load_state_dict({"sf": ck["sf"], "si": ck["si"]})
        if "spawn_rng" in ck:
            self._rng_state.copy_(ck["spawn_rng"])
            self._spawn_nodes.copy_(ck["last_spawn"])
            self._seeded = True
        if "done_flags" in ck and self.autoreset:
            self.done_flags.copy_(ck["done_flags"])
        self.render_obs()
        if self.bev is not None:
            self.render_bev()

    def load_state_dict(self, state: Dict[str, torch.Tensor]):
        with torch.cuda.device(self.device):
            sf = state["sf"].to(device=self.device, dtype=torch.float64).contiguous()
            si = state["si"].to(device=self.device, dtype=torch.int32).contiguous()
            _lib.check(self._L.tc_set_state(self._h, _ptr(sf), _ptr(si), self._stream()), "tc_set_state")
            torch.cuda.current_stream(self.device).synchronize()
        self._was_reset = True

    def profile_begin(self, max_steps: int):
        _lib.check(self._L.tc_profile_begin(self._h, int(max_steps)), "tc_profile_begin")

    def profile_end(self):
        """-> ({"track": ms, "project": ms, "raster": ms} summed over the recorded steps, number of steps)"""
        ms = (C.c_double * 3)()
        n = C.c_int32()
        _lib.check(self._L.tc_profile_end(self._h, ms, C.byref(n)), "tc_profile_end")
        return {"track": ms[0], "project": ms[1], "raster": ms[2]}, int(n.value)

    def cull_info(self) -> Dict[str, float]:
        """Visible-set tables of the small-frame render kernel (tc_debug_cull_info): camera reach they were built for
        (-1: culling off, -2: per-class rendering without such tables), cell count, mean / max nodes per cell."""
        out = (C.c_double * 4)()
        _lib.check(self._L.tc_debug_cull_info(self._h, out), "tc_debug_cull_info")
        return {"radius": out[0], "cells": int(out[1]), "mean_nodes": out[2], "max_nodes": int(out[3])}

    def render_info(self) -> Dict[str, int]:
        """Which kernels this env launches (tc_debug_render_info): block-per-env render path, envs per block of the packed
        kernel, its primitive chunks, the render kernel's dynamic shared memory, thread-per-env tracking."""
        out = (C.c_int32 * 8)()
        _lib.check(self._L.tc_debug_render_info(self._h, out), "tc_debug_render_info")
        keys = ("block_per_env", "envs_per_block", "prim_chunks", "render_smem", "track_per_thread", "banded_smem", "cell_nodes_cap", "cell_bytes_cap")
        d = dict(zip(keys, (int(v) for v in out)))
        v = d["track_per_thread"]
        d["track_per_thread"], d["blocks_per_sm"], d["track_lanes_per_env"] = v & 1, (v >> 4) & 63, 1 if v & 1 else v >> 10
        return d

    def cull_stats(self) -> Dict[str, float]:
        """Visible-set table bookkeeping: host builds, cache hits, milliseconds of the last / of all builds."""
        out = (C.c_double * 4)()
        _lib.check(self._L.tc_debug_cull_stats(self._h, out), "tc_debug_cull_stats")
        return {"builds": int(out[0]), "cache_hits": int(out[1]), "last_build_ms": out[2], "total_build_ms": out[3]}

    @property
    def launch_count(self) -> int:
        return int(self._L.tc_launch_count(self._h))

    def debug_layer_query(self, op: int, pos=(0.0, 0.0), angle: float = 0.0, edge=(0, 0)):
        """Test hook: a layer.py query evaluated by the device functions on class 0 (tc_debug_layer_query)."""
        with torch.cuda.device(self.device):
            oi = torch.zeros(1, dtype=torch.int32, device=self.device)
            od = torch.zeros(1, dtype=torch.float64, device=self.device)
            _lib.check(self._L.tc_debug_layer_query(self._h, op, float(pos[0]), float(pos[1]), float(angle), int(edge[0]), int(edge[1]),
                                                    _ptr(oi), _ptr(od), self._stream()), "tc_debug_layer_query")
            return int(oi.item()), float(od.item())
