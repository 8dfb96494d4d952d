"""Configuration loading with the reference's schema and defaults (tinycarlo/env.py:27-45, car.py:12-18,
camera.py:16-21, map.py:13-17). A config is a path to a .yaml file, a directory holding config.yaml, or a dict with
the mandatory sections sim / car / camera / map (a missing section raises KeyError, as in the reference)."""
import math
import numbers
import os
from typing import Any, Dict, List, Optional, Tuple, Union

import numpy as np

MAPS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "maps")


def load_config(config: Optional[Union[str, Dict[str, Any]]]) -> Tuple[Dict[str, Any], Optional[str]]:
    """Returns (config dict, absolute path of the yaml file or None). env.py:27-35."""
    config_path = None
    if isinstance(config, str):
        import yaml
        if config.endswith(".yaml"):
            config_path = os.path.abspath(config)
        else:
            config_path = os.path.abspath(os.path.join(config, "config.yaml"))
        with open(config_path, "r") as stream:
            config = yaml.safe_load(stream)
    if config is None:
        raise TypeError("config must be a yaml path, a directory with config.yaml, or a dict")
    for section in ("sim", "car", "camera", "map"):
        config[section]  # KeyError like the reference
    return config, config_path


def resolve_map_path(map_config: Dict[str, Any], config_path: Optional[str]) -> str:
    """map.py:15-16: json_path is relative to the yaml's directory, or to the CWD for dict configs. As an extension,
    {"map_name": "knuffingen"} selects one of the maps bundled in tinycarlo_b200/maps/."""
    if "map_name" in map_config and "json_path" not in map_config:
        return os.path.join(MAPS_DIR, map_config["map_name"] + ".json")
    base = "./" if config_path is None else os.path.dirname(config_path)
    return os.path.join(base, map_config["json_path"])


def sim_params(config: Dict[str, Any]) -> Dict[str, Any]:
    sim = config["sim"]
    fps = sim.get("fps", 30)
    return {"fps": fps, "T": 1 / fps, "observation_space_format": sim.get("observation_space_format", "rgb"),
            "render_realtime": sim.get("render_realtime", False),
            "overview_pixel_per_meter": sim.get("overview_pixel_per_meter", 150),
            "render_node_names": sim.get("render_node_names", False)}


def car_param_row(car_config: Dict[str, Any], T: float):
    """One row of the per-env car parameter table (include/tinycarlo_b200.h TC_CP_*); None -> NaN (car.py:12-18)."""
    def g(key, default):
        v = car_config.get(key, default)
        return math.nan if v is None else float(v)
    if car_config.get("max_acceleration", None) is not None and car_config.get("max_deceleration", None) is None:
        # car.py:82 would raise TypeError on `None * dt`
        raise TypeError("car.max_deceleration must be set when car.max_acceleration is set")
    return [g("wheelbase", 0.08), g("track_width", 0.03), g("max_velocity", 1), g("max_steering_angle", 35),
            g("steering_speed", None), g("max_acceleration", None), g("max_deceleration", None), float(T)]


LINE_THICKNESS_MAX = 255   # the rasteriser's 16.16 fixed-point set-up needs max(H, W) + 2 * thickness < 2^15


def is_line_thickness(t) -> bool:
    """camera line thickness: an integer in 1..LINE_THICKNESS_MAX (cv2.polylines rejects 0 and negative values)"""
    return isinstance(t, numbers.Integral) and not isinstance(t, bool) and 1 <= t <= LINE_THICKNESS_MAX


def camera_params(camera_config: Dict[str, Any]) -> Dict[str, Any]:
    """camera.py:16-21 defaults. max_range=None crashes the reference on the first frame (camera.py:80-82, SURVEY
    section 5); it is rejected here at construction, as is a line_thickness outside 1..255."""
    cam = {"resolution": list(camera_config.get("resolution", [128, 160])),
           "position": list(camera_config.get("position", [0, 0, 0])),
           "orientation": list(camera_config.get("orientation", [0, 0, 0])),
           "fov": camera_config.get("fov", 90),
           "max_range": camera_config.get("max_range", None),
           "line_thickness": camera_config.get("line_thickness", 1)}
    if not cam["max_range"]:
        raise ValueError("camera.max_range must be a positive number (the reference raises on the first frame when it is None)")
    if not is_line_thickness(cam["line_thickness"]):
        raise ValueError(f"camera.line_thickness must be an integer in 1..{LINE_THICKNESS_MAX}, got {cam['line_thickness']!r}")
    cam["line_thickness"] = int(cam["line_thickness"])
    return cam


RIG_KEYS = ("position", "orientation", "fov", "max_range", "line_thickness")


def camera_rig(config: Dict[str, Any]) -> Optional[List[Dict[str, Any]]]:
    """The optional top-level `cameras` list (an extension: several cameras per car, include/tinycarlo_b200.h tc_create_rig):
    one camera_params() section per entry, each the config's `camera` section with the entry's keys overriding it ({} is that
    camera itself), or None when the config has no such key. All cameras share camera.resolution: an entry with its own
    resolution raises ValueError, as do unknown keys (per-camera resolutions are what TinyCarloGroupedVecEnv's groups are for)."""
    rig = config.get("cameras")
    if rig is None:
        return None
    if not isinstance(rig, list) or not rig:
        raise ValueError(f"cameras must be a non-empty list of mappings, got {rig!r}")
    out = []
    for k, entry in enumerate(rig):
        if not isinstance(entry, dict):
            raise ValueError(f"cameras[{k}] must be a mapping, got {entry!r}")
        if "resolution" in entry:
            raise ValueError(f"cameras[{k}]: all cameras share camera.resolution (use TinyCarloGroupedVecEnv for several resolutions)")
        unknown = sorted(set(entry) - set(RIG_KEYS))
        if unknown:
            raise ValueError(f"cameras[{k}]: unknown keys {unknown} (allowed: {list(RIG_KEYS)})")
        merged = dict(config["camera"])
        merged.update(entry)
        out.append(camera_params(merged))
    return out


BEV_MAX_CLASSES = 16              # TC_MAX_CLASSES: planes of one BEV
BEV_SMEM_MAX = 200 * 1024         # TC_BEV_SMEM_MAX: shared memory of the BEV kernel's stacked bit plane
BEV_FORMATS = ("classes", "classes_bits")


def bev_params(config: Dict[str, Any], n_classes: int) -> Optional[Dict[str, Any]]:
    """The optional `bev` section (an extension: an ego-centric bird's-eye view of the lanes, include/tinycarlo_b200.h
    tc_set_bev) with its defaults, or None when the config has none. Raises ValueError for a bad section."""
    bev = config.get("bev")
    if bev is None:
        return None
    if not isinstance(bev, dict):
        raise ValueError("bev must be a mapping")

    def integer(v):
        return isinstance(v, numbers.Integral) and not isinstance(v, bool)

    def finite(v):
        return isinstance(v, numbers.Real) and not isinstance(v, bool) and math.isfinite(v)
    res = bev.get("resolution", [128, 128])
    if not (isinstance(res, (list, tuple)) and len(res) == 2 and all(integer(v) for v in res)
            and all(0 < v <= 4096 for v in res)):
        raise ValueError(f"bev.resolution must be [H, W] with integers in 1..4096, got {res!r}")
    H, W = int(res[0]), int(res[1])
    ppm = bev.get("pixel_per_meter", 128)
    if not (finite(ppm) and ppm > 0):
        raise ValueError(f"bev.pixel_per_meter must be a finite number > 0, got {ppm!r}")
    car = bev.get("car_pixel", [W / 2, 7 * H / 8])
    if not (isinstance(car, (list, tuple)) and len(car) == 2 and all(finite(v) for v in car)):
        raise ValueError(f"bev.car_pixel must be [col, row] with finite numbers, got {car!r}")
    t = bev.get("line_thickness", 1)
    if not (integer(t) and 1 <= t <= 8):
        raise ValueError(f"bev.line_thickness must be an integer in 1..8, got {t!r}")
    route = bev.get("route", False)
    if not isinstance(route, bool):
        raise ValueError(f"bev.route must be true or false, got {route!r}")
    fmt = bev.get("format", "classes")
    if fmt not in BEV_FORMATS:
        raise ValueError(f"bev.format must be one of {BEV_FORMATS}, got {fmt!r}")
    if fmt == "classes_bits" and (H * W) % 32 != 0:
        raise ValueError("bev.format classes_bits needs H*W to be a multiple of 32")
    planes = n_classes + int(route)
    if planes > BEV_MAX_CLASSES:
        raise ValueError(f"bev: {planes} planes (classes + route) exceed {BEV_MAX_CLASSES}")
    words = (planes * H * W + 31) // 32 + 1
    if (words * 4 + 15) // 16 * 16 > BEV_SMEM_MAX:
        raise ValueError(f"bev: {planes} planes of {H}x{W} do not fit the kernel's shared memory ({BEV_SMEM_MAX} bytes of bit planes)")
    return {"resolution": [H, W], "pixel_per_meter": float(ppm), "car_pixel": [float(car[0]), float(car[1])], "line_thickness": int(t),
            "route": route, "format": fmt, "planes": planes}


LIDAR_MAX_RAYS = 1024             # TC_LIDAR_RPT * TC_LIDAR_THREADS: rays of one scan


def lidar_params(config: Dict[str, Any], n_classes: int) -> Optional[Dict[str, Any]]:
    """The optional `lidar` section (an extension: a range scan of R rays around every car, per laneline class the distance
    to the first edge along each ray, include/tinycarlo_b200.h tc_set_lidar) with its defaults, or None when the config has
    none. Raises ValueError for a bad section."""
    lidar = config.get("lidar")
    if lidar is None:
        return None
    if not isinstance(lidar, dict):
        raise ValueError("lidar must be a mapping")
    unknown = sorted(set(lidar) - {"rays", "fov", "max_range", "origin"})
    if unknown:
        raise ValueError(f"lidar: unknown keys {unknown} (allowed: rays, fov, max_range, origin)")

    def finite(v):
        return isinstance(v, numbers.Real) and not isinstance(v, bool) and math.isfinite(v)
    rays = lidar.get("rays", 64)
    if not (isinstance(rays, numbers.Integral) and not isinstance(rays, bool) and 1 <= rays <= LIDAR_MAX_RAYS):
        raise ValueError(f"lidar.rays must be an integer in 1..{LIDAR_MAX_RAYS}, got {rays!r}")
    fov = lidar.get("fov", 360)
    if not (finite(fov) and 0 < fov <= 360):
        raise ValueError(f"lidar.fov must be a number of degrees in (0, 360], got {fov!r}")
    max_range = lidar.get("max_range", 0.5)
    if not (finite(max_range) and max_range > 0):
        raise ValueError(f"lidar.max_range must be a finite number > 0 (metres), got {max_range!r}")
    origin = lidar.get("origin", [0.0, 0.0])
    if not (isinstance(origin, (list, tuple)) and len(origin) == 2 and all(finite(v) for v in origin)):
        raise ValueError(f"lidar.origin must be [forward, right] with finite numbers (metres), got {origin!r}")
    return {"rays": int(rays), "fov": float(fov), "max_range": float(max_range), "origin": [float(origin[0]), float(origin[1])],
            "classes": int(n_classes)}


NAV_MAX_GOALS = 4096             # tc_set_route: goal candidates of one handle


def navigation_params(config: Dict[str, Any], tables) -> Optional[Dict[str, Any]]:
    """The optional `navigation` section (an extension: a goal node per car with the route's next maneuver, the distance left
    and the progress along it, include/tinycarlo_b200.h tc_set_route) with its defaults, or None when the config has none.
    tables: the map's MapTables. Keys: goals (lanepath node ids; default the map's spawn_points that have an incoming
    lanepath edge, else every node with one), reach_radius (metres, default 0.05), on_reach ("resample", the default, or "terminate"). Raises ValueError
    for a bad section."""
    nav = config.get("navigation")
    if nav is None:
        return None
    if not isinstance(nav, dict):
        raise ValueError("navigation must be a mapping")
    unknown = sorted(set(nav) - {"goals", "reach_radius", "on_reach"})
    if unknown:
        raise ValueError(f"navigation: unknown keys {unknown} (allowed: goals, reach_radius, on_reach)")
    n_nodes = len(tables.lp_nodes)
    has_pred = np.zeros(n_nodes, bool)
    has_pred[tables.lp_edges[:, 1]] = True
    goals = nav.get("goals")
    if goals is None:
        # the spawn points a car can arrive at (a spawn node without an incoming edge is only ever a start)
        goals = [g for g in tables.spawn_points if has_pred[g]] if tables.spawn_points is not None else \
            [int(v) for v in np.nonzero(has_pred)[0]]
    if not (isinstance(goals, (list, tuple)) and 1 <= len(goals) <= NAV_MAX_GOALS
            and all(isinstance(g, numbers.Integral) and not isinstance(g, bool) for g in goals)):
        raise ValueError(f"navigation.goals must be a list of 1..{NAV_MAX_GOALS} lanepath node ids, got {goals!r}")
    for g in goals:
        if not 0 <= g < n_nodes:
            raise ValueError(f"navigation.goals: node {g} is not a lanepath node (0..{n_nodes - 1})")
        if not has_pred[g]:
            raise ValueError(f"navigation.goals: node {g} has no incoming lanepath edge, so no car can reach it")
    reach = nav.get("reach_radius", 0.05)
    if not (isinstance(reach, numbers.Real) and not isinstance(reach, bool) and math.isfinite(reach) and reach >= 0):
        raise ValueError(f"navigation.reach_radius must be a finite number >= 0 (metres), got {reach!r}")
    on_reach = nav.get("on_reach", "resample")
    if on_reach not in ("resample", "terminate"):
        raise ValueError(f"navigation.on_reach must be 'resample' or 'terminate', got {on_reach!r}")
    return {"goals": [int(g) for g in goals], "reach_radius": float(reach), "on_reach": on_reach}


# ------------------------------------------------------------------------------------------------ shipped configurations
# The car / camera sections of examples/config_knuffingen.yaml and config_simple_layout.yaml, and the spawn points they
# list, as dict configs over the maps bundled in tinycarlo_b200/maps/ (benchmarks, tools and tests build theirs from these).
CAR_SHIPPED = {"wheelbase": 0.0487, "track_width": 0.027, "max_velocity": 0.1, "max_steering_angle": 30, "steering_speed": 30,
               "max_acceleration": 0.1, "max_deceleration": 1.0}
CAM_SHIPPED = {"position": [0.0, -0.005, 0.04], "orientation": [22, 0, 0], "resolution": [128, 160], "fov": 80, "max_range": 0.5,
               "line_thickness": 2}
SPAWN_KNUFF = [156, 18, 217, 214, 325, 354, 176, 402, 339, 376, 385, 419, 396, 37, 149, 62, 240, 113, 98, 299, 2]
SPAWN_SIMPLE = [57, 143, 112, 121, 138, 157, 67, 46, 165, 124, 79, 33, 84, 21, 178, 7]
PPM = {"knuffingen": 222, "simple_layout": 450, "formula_student_track": 300, "formula_student_skidpad": 200}


def make_config(map_name: str, fmt: str, car: Optional[Dict[str, Any]] = None, cam: Optional[Dict[str, Any]] = None, spawn="default",
                fps: int = 30) -> Dict[str, Any]:
    """Dict config on a bundled map: the shipped car / camera sections with `car` / `cam` overrides. spawn: "default" (the
    yaml's spawn_points for knuffingen / simple_layout), None (any node with a successor, map.py:51-69) or a node list."""
    car_cfg = dict(CAR_SHIPPED)
    car_cfg.update(car or {})
    cam_cfg = {k: (list(v) if isinstance(v, list) else v) for k, v in CAM_SHIPPED.items()}
    cam_cfg.update(cam or {})
    map_cfg = {"map_name": map_name, "pixel_per_meter": PPM[map_name]}
    if spawn == "default":
        if map_name == "knuffingen":
            map_cfg["spawn_points"] = list(SPAWN_KNUFF)
        elif map_name == "simple_layout":
            map_cfg["spawn_points"] = list(SPAWN_SIMPLE)
    elif spawn is not None:
        map_cfg["spawn_points"] = list(spawn)
    return {"sim": {"fps": fps, "observation_space_format": fmt}, "car": car_cfg, "camera": cam_cfg, "map": map_cfg}
