"""CPU checks of the bird's-eye view: the host build of tc_bev_segment + the lane-group rasteriser (tc_core.cuh, what
tc_bev_kernel runs) against the numpy + cv2.polylines restatement of the contract, and the validation of the config's
`bev` section."""
import math

import numpy as np
import pytest

import map_shapes_util as MS
from bev_util import host_bev as bev
from bev_util import oracle_bev
from hosttest_util import HostCore
from tinycarlo_b200.config import MAPS_DIR, PPM, bev_params, make_config
from tinycarlo_b200.maptables import MapTables

cv2 = pytest.importorskip("cv2")

# the bundled maps (5 or 3 classes) and Knuffingen regrouped into 1, 2, 15 and 16 classes (tests/map_shapes_util.py)
MAPS = ["knuffingen", "simple_layout", "formula_student_track", "formula_student_skidpad", "K1", "K2", "K15", "K16", "K16R"]
# (resolution, car pixel, thickness, route, pixel_per_meter)
CASES = [((128, 128), "default", 1, False, 128.0),
         ((64, 64), "centre", 2, True, 40.0),
         ((96, 128), "bottom", 3, True, 100.0),
         ((75, 100), "outside", 6, False, 60.0),
         ((128, 128), "default", 8, True, 25.0),
         ((75, 100), "centre", 1, True, 150.0),
         # thickness
         ((128, 128), "default", 4, True, 128.0),
         ((128, 128), "negative", 5, True, 128.0),
         ((128, 128), "default", 7, False, 128.0),
         # planes that start part-way into a word; extreme aspect ratios
         ((33, 35), "default", 2, True, 60.0),
         ((129, 129), "centre", 4, True, 128.0),
         ((1, 1), "centre", 3, True, 128.0),
         ((1, 4096), "default", 2, True, 128.0),
         ((4096, 1), "default", 5, True, 128.0),
         ((7, 1001), "default", 5, False, 200.0),
         # scale: the whole map in a few pixels up to endpoints beyond int32 (INT_MIN)
         ((128, 128), "default", 3, True, 2.0),
         ((128, 128), "bottom", 4, True, 1000.0),
         ((128, 128), "centre", 2, True, 1e6),
         ((128, 128), "default", 8, True, 1e9)]


def car_pixel(kind, H, W):
    return {"default": (W / 2, 7 * H / 8), "centre": (W / 2, H / 2), "bottom": (W / 2 - 3.5, H - 1.0), "outside": (-12.25, H + 20.0),
            "negative": (-3.75, -0.5)}[kind]


def load_tables(map_name, directory):
    if map_name in MS.MAPS:
        return MapTables(MS.write(MS.MAPS[map_name](), directory, map_name), MS.PPM)
    return MapTables(f"{MAPS_DIR}/{map_name}.json", PPM[map_name])


@pytest.fixture(scope="module")
def map_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("maps")


def poses(tables, rng, n):
    """n states: on the map (near lanepath nodes, or exactly on a laneline node, where that node's edges pass through the car
    pixel at any scale) and off it, any heading, with local paths of 0-4 lanepath edges"""
    sf = np.zeros((n, 8))
    si = np.full((n, 16), -1, np.int32)
    lo, hi = tables.ll_nodes.min(0), tables.ll_nodes.max(0)
    for i in range(n):
        if i % 4 == 3:   # off the map
            sf[i, :2] = hi + rng.uniform(0.2, 3.0, 2) * rng.choice([-1, 1], 2) + (lo - hi) * (rng.random() < 0.5)
        elif i % 4 == 1:
            sf[i, :2] = tables.ll_nodes[rng.integers(len(tables.ll_nodes))]
        else:
            sf[i, :2] = tables.lp_nodes[rng.integers(len(tables.lp_nodes))] + rng.normal(0, 0.05, 2)
        sf[i, 2] = rng.uniform(-math.pi, math.pi) if i % 5 else rng.uniform(-40, 40)   # headings beyond +-pi too
        plen = int(rng.integers(0, 5))
        si[i, 0] = plen
        for j in range(plen):
            si[i, 2 + 2 * j:4 + 2 * j] = tables.lp_edges[rng.integers(len(tables.lp_edges))]
    return sf, si


@pytest.mark.parametrize("map_name", MAPS)
@pytest.mark.parametrize("case", range(len(CASES)))
def test_host_bev_matches_cv2_oracle(map_name, case, map_dir):
    (H, W), kind, t, route, ppm = CASES[case]
    tables = load_tables(map_name, map_dir)
    core = HostCore(tables, 1, np.zeros(8), np.zeros(20), 1, 8, 8)
    rng = np.random.default_rng(1000 * case + len(map_name))
    sf, si = poses(tables, rng, 12)
    cp = car_pixel(kind, H, W)
    got = bev(core, sf, si, H, W, ppm, cp, t, route)
    assert got.shape == (12, tables.n_classes + int(route), H, W)
    drawn = 0
    for i in range(12):
        want = oracle_bev(tables, sf[i], si[i], H, W, ppm, cp, t, route)
        assert np.array_equal(got[i], want), (map_name, CASES[case], i, np.argwhere(got[i] != want)[:5])
        drawn += int(want.any())
    # the poses on the map see lanes; in a 1x1 frame or at 1e6 px/m and more, only those exactly on a laneline node do
    assert drawn >= (3 if H * W == 1 or ppm >= 1e6 else 4)


def test_host_bev_orientation():
    """the car points up, its right is image right: a lane 0.2 m ahead is above the car pixel, one 0.2 m to the right is right of it"""
    tables = MapTables(f"{MAPS_DIR}/simple_layout.json", PPM["simple_layout"])
    core = HostCore(tables, 1, np.zeros(8), np.zeros(20), 1, 8, 8)
    # heading +x (rot 0): in image-like map coordinates (y down) the car's right is +y
    node = tables.class_nodes(0)[0]
    sf = np.zeros((2, 8))
    sf[0, :3] = [node[0] - 0.2, node[1], 0.0]   # node straight ahead
    sf[1, :3] = [node[0], node[1] - 0.2, 0.0]   # node to the right
    out = bev(core, sf, np.zeros((2, 16), np.int32), 129, 129, 100.0, (64, 64), 1)
    ys, xs = np.nonzero(out[0, 0])
    assert np.any((ys == 64 - 20) & (xs == 64))
    ys, xs = np.nonzero(out[1, 0])
    assert np.any((ys == 64) & (xs == 64 + 20))


def cfg_with(bev, map_name="simple_layout"):
    c = make_config(map_name, "classes")
    c["bev"] = bev
    return c


def test_bev_params_defaults():
    assert bev_params(make_config("knuffingen", "classes"), 5) is None
    p = bev_params(cfg_with({}), 5)
    assert p == {"resolution": [128, 128], "pixel_per_meter": 128.0, "car_pixel": [64.0, 112.0], "line_thickness": 1, "route": False,
                 "format": "classes", "planes": 5}
    p = bev_params(cfg_with({"resolution": [75, 100], "route": True, "format": "classes", "line_thickness": 8}), 5)
    assert p["car_pixel"] == [50.0, 75 * 7 / 8] and p["planes"] == 6
    assert bev_params(cfg_with({"resolution": [64, 96], "format": "classes_bits", "car_pixel": [-3, 200.5]}), 3)["car_pixel"] == [-3.0, 200.5]


@pytest.mark.parametrize("bad", [
    {"resolution": [0, 128]}, {"resolution": [128, -4]}, {"resolution": [128.5, 128]}, {"resolution": [128]},
    {"resolution": [float("inf"), 128]}, {"pixel_per_meter": 0}, {"pixel_per_meter": -3.0}, {"pixel_per_meter": float("nan")},
    {"pixel_per_meter": float("inf")}, {"car_pixel": [float("nan"), 3]}, {"car_pixel": [1]},
    {"line_thickness": 0}, {"line_thickness": 9}, {"line_thickness": 2.5},
    {"format": "rgb"}, {"format": "classes_bf16"}, {"format": "classes_bits", "resolution": [75, 100]},
    {"route": "yes"}, {"resolution": [1024, 512]}, {"resolution": [4096, 4096]}, {"resolution": [512, 534], "route": True},
])
def test_bev_params_rejects(bad):
    with pytest.raises(ValueError):
        bev_params(cfg_with(bad), 5)


def test_bev_params_rejects_too_many_planes():
    assert bev_params(cfg_with({"route": True}), 15)["planes"] == 16
    with pytest.raises(ValueError):
        bev_params(cfg_with({"route": True}), 16)
    with pytest.raises(ValueError):
        bev_params(cfg_with({}), 17)


def test_bev_params_shared_memory_bound():
    """the largest stacked planes that fit the kernel's 200 KB (P*H*W bits + a pad word, rounded up to 16 bytes): 6 planes of
    512x533 (204 688 B) and 16 of 316x324 (204 784 B); one column more is rejected"""
    assert bev_params(cfg_with({"resolution": [512, 533], "route": True}), 5)["planes"] == 6
    assert bev_params(cfg_with({"resolution": [316, 324], "route": True}), 15)["planes"] == 16
    with pytest.raises(ValueError, match="shared memory"):
        bev_params(cfg_with({"resolution": [316, 325], "route": True}), 15)
