"""TinyCarloEnv — single-environment drop-in for the reference's gymnasium env (tinycarlo/env.py:15-147), a batch of one
on the CUDA path.

    env = gym.make("tinycarlo-v2", config="config.yaml")          # when gymnasium is installed
    env = tinycarlo_b200.TinyCarloEnv(config={...})                # always

Same constructor arguments, action dict, observation array, `info` dict layout, default reward / termination and
`truncated` semantics as the reference, and the attributes its wrappers and examples touch (`unwrapped.wrapped`,
`.car.track_width`, `.observation_space_format`, `.no_observation`, `.camera.orientation/.fov/.update_params()`,
`.config`, `.render_mode`, `.map.get_laneline_names()`). Observations and info values come back as numpy / Python
objects; the numbers are the float64 state of the kernels. `render_mode="human"` shows the camera frame and the bird's-eye
overview (tinycarlo_b200/overview.py) in OpenCV windows like the reference; `render_overview()` returns that image."""
from typing import Any, Dict, Optional, Tuple, Union

import numpy as np
import torch

from . import gym_compat as gc
from .vec_env import TinyCarloVecEnv


class _CarFacade:
    """The attributes of tinycarlo.car.Car that the reference's wrappers / examples read."""

    def __init__(self, env: "TinyCarloEnv"):
        self._env = env
        cfg = env.config["car"]
        self.track_width = cfg.get("track_width", 0.03)
        self.wheelbase = cfg.get("wheelbase", 0.08)
        self.max_velocity = cfg.get("max_velocity", 1)
        self.max_steering_angle = cfg.get("max_steering_angle", 35)
        self.steering_speed = cfg.get("steering_speed", None)
        self.max_acceleration = cfg.get("max_acceleration", None)
        self.max_deceleration = cfg.get("max_deceleration", None)
        self.T = env.T

    def _state(self):
        st = self._env._vec.state_dict()
        return st["sf"][0].cpu().numpy(), st["si"][0].cpu().numpy()

    @property
    def position(self):
        sf, _ = self._state()
        return [float(sf[0]), float(sf[1])]

    @property
    def position_front(self):
        sf, _ = self._state()
        return (float(sf[5]), float(sf[6]))

    @property
    def rotation(self):
        return float(self._state()[0][2])

    @property
    def steering_angle(self):
        return float(self._state()[0][3])

    @property
    def velocity(self):
        return float(self._state()[0][4])

    @property
    def local_path(self):
        _, si = self._state()
        return [(int(si[2 + 2 * i]), int(si[3 + 2 * i])) for i in range(int(si[0]))]

    @property
    def last_maneuver(self):
        return int(self._state()[1][1])


class _CameraFacade:
    """tinycarlo.camera.Camera's mutable parameters; update_params() re-stages E and K (camera.py:48-50). With a camera rig
    (the config's `cameras` list) there is one facade per camera, `index` m."""

    def __init__(self, env: "TinyCarloEnv", index: int = 0):
        self._env = env
        self.index = index
        cc = env._vec.cam_cfgs[index]
        self.resolution = list(cc["resolution"])
        self.position = list(cc["position"])
        self.orientation = list(cc["orientation"])
        self.fov = cc["fov"]
        self.max_range = cc["max_range"]
        self.line_thickness = cc["line_thickness"]

    def _view(self, t):
        """this camera's frame of env 0 in a tensor of the vec env's layout"""
        return t[0] if self._env._vec.rig is None else t[0, self.index]

    def update_params(self):
        v = self._env._vec
        v.set_camera_params(position=np.asarray(self.position, np.float64), orientation=np.asarray(self.orientation, np.float64),
                            fov=float(self.fov), max_range=float(self.max_range), line_thickness=int(self.line_thickness),
                            camera=None if v.rig is None else self.index)

    @property
    def E(self):
        return self._env._vec._cam_rows[self.index, :12].reshape(3, 4).copy()

    @property
    def K(self):
        r = self._env._vec._cam_rows[self.index]
        return np.array([[r[12], 0, r[14]], [0, r[13], r[15]], [0, 0, 1]])

    def get_last_frame_rgb(self):
        return self._view(self._env._vec.render_rgb()).cpu().numpy()

    def get_last_frame_classes(self):
        if self._env.observation_space_format == "rgb":
            return None
        return self._view(self._env._vec.obs).cpu().numpy().copy()


class TinyCarloEnv(gc.Env):
    metadata: Dict[str, list] = {"render_modes": ["human", "rgb_array"]}

    def __init__(self, render_mode: Optional[str] = None, config: Optional[Union[str, Dict[str, Any]]] = None, device="cuda"):
        self._vec = TinyCarloVecEnv(config, 1, device=device)
        v = self._vec
        self.config, self.config_path = v.config, v.config_path
        self.fps, self.T = v.fps, v.T
        self.observation_space_format: str = v.observation_space_format
        self.map = v.map
        self.car = _CarFacade(self)
        # camera rig: one facade per camera; `camera` is camera 0, the reference's one camera
        self.cameras = [_CameraFacade(self, m) for m in range(v.n_cameras)]
        self.camera = self.cameras[0]
        self._wrapped = False
        self._overview = None
        self._windows = None
        assert render_mode is None or render_mode in self.metadata["render_modes"]
        self.render_mode = render_mode
        self.no_observation = False
        self.action_space = gc.spaces.Dict({"car_control": gc.spaces.Box(-1, 1, shape=(2,), dtype=np.float32),
                                            "maneuver": gc.spaces.Discrete(4)})
        self.observation_space = gc.spaces.Box(low=0, high=255, shape=tuple(v.obs_shape), dtype=np.uint8)
        self._cc = torch.zeros((1, 2), dtype=torch.float64, device=v.device)
        self._man = torch.zeros(1, dtype=torch.int32, device=v.device)
        self.reset()

    # env.py:53,137-138: wrappers set `unwrapped.wrapped = True` to switch the default reward/termination off
    @property
    def wrapped(self) -> bool:
        return self._wrapped

    @wrapped.setter
    def wrapped(self, value: bool):
        self._wrapped = bool(value)
        self._vec.set_wrapped(self._wrapped)

    def invalidate_obs(self):
        """TinyCarloVecEnv.invalidate_obs of the one-env vector env behind this env."""
        self._vec.invalidate_obs()

    def _sync_flags(self):
        # env.py:77-81: observations are skipped only when no_observation is set and there is no render mode
        self._vec.no_observation = bool(self.no_observation and self.render_mode is None)

    def _obs(self) -> np.ndarray:
        if self._vec.no_observation:
            return np.zeros(self.observation_space.shape, dtype=np.uint8)
        return self._vec.obs[0].cpu().numpy().copy()

    def _info(self) -> Dict[str, Any]:
        v = self._vec
        i64 = v.out["info_f64"][0].cpu().numpy()
        sf = v.state_dict()["sf"][0].cpu().numpy()
        plen = int(v.out["path_len"][0].item())
        names = v.class_names
        nodes = v.out["local_path_nodes"][0].cpu().numpy()
        if plen >= 2:   # car.py:47-51: shorter paths give the empty info
            local_path = [[float(x) for x in v.map.lp_nodes[int(nodes[i, 1])]] for i in range(plen)]
            dist = {n: float(i64[4 + k]) for k, n in enumerate(names)}
            cte, he, vel = float(i64[0]), float(i64[1]), float(i64[2])
        else:
            local_path, dist, cte, he, vel = [], {n: 0 for n in names}, 0, 0, 0.0
        info = {"cte": cte, "heading_error": he, "position": [float(sf[0]), float(sf[1])], "orientation": float(sf[2]),
                "laneline_distances": dist, "local_path": local_path, "velocity": vel}
        if v.bev is not None:   # the config's `bev` section (an extension): this env's bird's-eye view
            info["bev"] = v.bev[0].cpu().numpy()
        if v.lidar is not None:   # the config's `lidar` section (an extension): this env's range scan [C, R]
            info["lidar"] = v.lidar[0].cpu().numpy()
        if v.route is not None:   # the config's `navigation` section (an extension): this env's goal and route
            r = v.route
            info.update({"goal": int(r["goal"][0].item()), "goal_position": [float(x) for x in r["goal_position"][0].cpu().numpy()],
                         "route_command": int(r["command"][0].item()), "route_distance": float(r["distance"][0].item()),
                         "route_progress": float(r["progress"][0].item()), "goal_reached": bool(r["reached"][0].item())})
        return info

    def reset(self, seed: Optional[int] = None, options: Optional[Any] = None) -> Tuple[np.ndarray, Dict[str, Any]]:
        super().reset(seed=seed)
        self._sync_flags()
        node = self.map.sample_spawn_node(self.np_random)   # map.py:51-69 on the env's own generator
        if not self._vec._seeded:
            self._vec._seed(0)   # the single env draws on the host generator gymnasium seeded; the device stream stays unused
        self._vec.reset(spawn_nodes=torch.tensor([node], dtype=torch.int32))
        if self.render_mode == "human":   # env.py:109-110: the reference shows its windows from reset() and step()
            self.render()
        return self._obs(), self._info()

    def step(self, action: Dict[str, Any]) -> Tuple[np.ndarray, float, bool, bool, Dict[str, Any]]:
        self._sync_flags()
        cc = np.clip(np.asarray(action["car_control"], dtype=np.float64), -1.0, 1.0)
        self._cc.copy_(torch.from_numpy(cc.reshape(1, 2)))
        self._man.fill_(int(action["maneuver"]))
        _, reward, terminated, truncated, _ = self._vec.step({"car_control": self._cc, "maneuver": self._man})
        i64 = self._vec.out["info_f64"][0, 3].item()
        rew = float(i64) if not self._wrapped else 0
        if self.render_mode == "human":   # env.py:140-141
            self.render()
        return self._obs(), rew, bool(terminated[0].item()), bool(truncated[0].item()), self._info()

    def render_overview(self) -> np.ndarray:
        """The map with the car and its tracked path on it (renderer.py:19-34), RGB uint8."""
        if self._overview is None:
            from .overview import OverviewRenderer
            sim = self.config["sim"]
            self._overview = OverviewRenderer(self.map, sim.get("overview_pixel_per_meter", 150), node_names=sim.get("render_node_names", False))
        sf, si = self.car._state()
        path = [(int(si[2 + 2 * i]), int(si[3 + 2 * i])) for i in range(max(int(si[0]), 0))]
        return self._overview.render([float(sf[0]), float(sf[1])], float(sf[2]), float(sf[3]), self.car.wheelbase, self.car.track_width, path)

    def render(self) -> Optional[np.ndarray]:
        """env.py:149-174: rgb_array -> the RGB camera frame (whatever the observation format; camera 0 of a rig); human -> two
        OpenCV windows"""
        if self.render_mode == "rgb_array":
            return self.camera.get_last_frame_rgb()
        if self.render_mode == "human":
            import cv2
            if self._windows is None:
                self._windows = ("Map", "Camera")
                for w in self._windows:
                    cv2.namedWindow(w, cv2.WINDOW_NORMAL | cv2.WINDOW_KEEPRATIO | cv2.WINDOW_GUI_NORMAL)
            cv2.imshow(self._windows[0], self.render_overview())
            cv2.imshow(self._windows[1], self.camera.get_last_frame_rgb())
            cv2.waitKey(max(int(self.T * 1000), 1) if self.config["sim"].get("render_realtime", False) else 1)
        return None

    def close(self):
        if self._windows is not None:
            import cv2
            for w in self._windows:
                cv2.destroyWindow(w)
            self._windows = None
        self._vec.close()
