"""CPU checks of the range scan: the host build of tc_lidar_stage + tc_lidar_hit (tc_core.cuh, what tc_lidar_kernel runs)
against the numpy restatement of the contract, bit for bit in float64; the cull's documented square; the validation of the
config's `lidar` section and of tc_set_lidar / tc_render_lidar."""
import ctypes as C
import math

import numpy as np
import pytest

import map_shapes_util as MS
from hosttest_util import HostCore
from lidar_util import SYN_LAYERS, SYN_RANGE, host_keep, host_lidar, oracle_lidar, synthetic_map
from tinycarlo_b200 import _lib
from tinycarlo_b200.config import MAPS_DIR, PPM, lidar_params, make_config
from tinycarlo_b200.maptables import MapTables

MAPS = ["knuffingen", "simple_layout", "formula_student_track", "formula_student_skidpad", "K1", "K2", "K15", "K16"]
# (rays, fov, max_range, origin [forward, right]): every R, fov and max_range of the contract's corners, origins offset
# forward, backward and sideways
SCANS = [(64, 360.0, 0.5, (0.0, 0.0)),
         (1, 360.0, 0.5, (0.1, 0.0)),
         (2, 90.0, 0.5, (-0.05, 0.0)),
         (3, 180.0, 1e6, (0.0, 0.03)),
         (1024, 360.0, 0.5, (0.0, -0.02)),
         (64, 1e-3, 1e6, (0.02, 0.01)),
         (64, 180.0, 1e-6, (0.0, 0.0)),
         (3, 90.0, 1e-6, (-0.03, -0.04)),
         (1024, 1e-3, 0.5, (0.0, 0.0)),
         (2, 360.0, 1e6, (0.2, -0.1))]


def load_tables(map_name, directory):
    if map_name in MS.MAPS:
        return MapTables(MS.write(MS.MAPS[map_name](), directory, map_name), MS.PPM)
    return MapTables(f"{MAPS_DIR}/{map_name}.json", PPM[map_name])


@pytest.fixture(scope="module")
def map_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("maps")


def poses(tables, rng, n):
    """n states: near lanepath nodes, exactly on a laneline node (distance +0.0 to the edges that meet there), off the map,
    and NaN; headings beyond +-pi too"""
    sf = np.zeros((n, 8))
    lo, hi = tables.ll_nodes.min(0), tables.ll_nodes.max(0)
    for i in range(n):
        if i % 6 == 5:
            sf[i, :3] = np.nan if i % 12 == 5 else [np.nan, 0.3, 0.1]
            continue
        if i % 4 == 3:   # off the map
            sf[i, :2] = hi + rng.uniform(0.2, 3.0, 2) * rng.choice([-1, 1], 2) + (lo - hi) * (rng.random() < 0.5)
        elif i % 4 == 1:
            sf[i, :2] = tables.ll_nodes[rng.integers(len(tables.ll_nodes))]
        else:
            sf[i, :2] = tables.lp_nodes[rng.integers(len(tables.lp_nodes))] + rng.normal(0, 0.05, 2)
        sf[i, 2] = rng.uniform(-math.pi, math.pi) if i % 5 else rng.uniform(-40, 40)
    return sf


@pytest.mark.parametrize("map_name", MAPS)
@pytest.mark.parametrize("scan", range(len(SCANS)))
def test_host_lidar_matches_oracle(map_name, scan, map_dir):
    rays, fov, max_range, origin = SCANS[scan]
    tables = load_tables(map_name, map_dir)
    core = HostCore(tables, 1, np.zeros(8), np.zeros(20), 1, 8, 8)
    rng = np.random.default_rng(100 * scan + len(map_name))
    n = 12
    sf = poses(tables, rng, n)
    got = host_lidar(core, sf, rays, fov, max_range, origin)
    assert got.shape == (n, tables.n_classes, rays)
    hits = 0
    for i in range(n):
        want = oracle_lidar(tables, sf[i], rays, fov, max_range, origin)
        assert np.array_equal(got[i].view(np.uint64), want.view(np.uint64)), (map_name, SCANS[scan], i, sf[i, :3],
                                                                             np.argwhere(got[i] != want)[:5])
        hits += int((want < max_range).any())
        if not np.isfinite(sf[i, :3]).all():
            assert (got[i] == max_range).all()
    if max_range >= 0.5:
        assert hits >= (2 if rays < 3 else 4)   # the poses on the map see lanes


def test_host_lidar_zero_is_positive_and_on_node(map_dir):
    """a car exactly on a laneline node is at distance +0.0 (never -0.0) from that node's class on (almost) every ray"""
    tables = load_tables("knuffingen", map_dir)
    core = HostCore(tables, 1, np.zeros(8), np.zeros(20), 1, 8, 8)
    sf = np.zeros((4, 8))
    for i in range(4):
        sf[i, :2] = tables.class_nodes(0)[7 * i + 3]
        sf[i, 2] = 0.4 * i - 1.0
    got = host_lidar(core, sf, 64, 360.0, 0.5)
    zeros = got[:, 0] == 0
    assert zeros.sum() >= 4 * 60
    assert not np.signbit(got[:, 0][zeros]).any()


@pytest.fixture(scope="module")
def synthetic(tmp_path_factory):
    return MapTables(synthetic_map(tmp_path_factory.mktemp("syn")), 1)


@pytest.mark.parametrize("rays,fov", [(1, 360.0), (3, 1e-3), (65, 90.0), (1023, 360.0), (5, 180.0)])
def test_host_lidar_synthetic_edge_cases(synthetic, rays, fov):
    """θ = 0 with odd R: ray (R-1)/2 is exactly (1, 0). u = 0 and u = 1 hit; t = 0 is +0.0; parallel, collinear and zero-length
    edges never hit; an edge at max_range gives max_range, as does one an ulp beyond; an edge that crosses the cull's square with
    both ends far outside it is seen; u an ulp either side of 1"""
    core = HostCore(synthetic, 1, np.zeros(8), np.zeros(20), 1, 8, 8)
    sf = np.zeros((1, 8))
    got = host_lidar(core, sf, rays, fov, SYN_RANGE)[0]
    want = oracle_lidar(synthetic, sf[0], rays, fov, SYN_RANGE)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    j = (rays - 1) // 2
    fwd = {name: got[p, j] for p, name in enumerate(SYN_LAYERS)}
    assert fwd["u0"] == pytest.approx(0.2, abs=1e-15) and fwd["u1"] == pytest.approx(0.15, abs=1e-15)
    assert fwd["zero"] == 0.0 and not np.signbit(fwd["zero"])
    for name in ("parallel", "collinear", "point", "at_range", "beyond"):
        assert fwd[name] == SYN_RANGE, name
    assert fwd["crossing"] == pytest.approx(0.1, abs=1e-15)
    assert fwd["near1_-3"] == fwd["near1_-2"] == pytest.approx(0.12, abs=1e-15)
    assert fwd["near1_2"] == fwd["near1_3"] == SYN_RANGE
    # the same cases as float32 words: what the device stores
    assert not np.signbit(got.astype(np.float32)).any()


def test_host_lidar_orientation(synthetic):
    """ray 0 looks left of the heading, ray R-1 right of it, and the car's right is (-sin, cos), as in the BEV: 9 rays over 180
    degrees are 20 degrees apart, from -80 (left) to +80 (right). The `zero` edge (x = 0, y in [-0.1, 0.1]) seen from
    (-0.05, 0) at heading +x is met by the rays within 63 degrees of the heading, symmetrically; with the origin 0.09 m to the
    right (+y) only the left rays still reach it."""
    core = HostCore(synthetic, 1, np.zeros(8), np.zeros(20), 1, 8, 8)
    zero = list(SYN_LAYERS).index("zero")
    sf = np.zeros((1, 8))
    sf[0, :2] = [-0.05, 0.0]
    got = host_lidar(core, sf, 9, 180.0, SYN_RANGE)[0, zero]
    assert got[4] == pytest.approx(0.05) and got[1] == pytest.approx(0.1) and got[7] == pytest.approx(0.1)
    assert got[0] == got[8] == SYN_RANGE
    got = host_lidar(core, sf, 9, 180.0, SYN_RANGE, origin=(0.0, 0.09))[0, zero]
    assert got[1] == pytest.approx(0.1) and got[4] == pytest.approx(0.05)
    assert got[0] == got[5] == got[7] == got[8] == SYN_RANGE


def test_lidar_cull_keeps_the_grown_square():
    """tc_lidar_stage keeps every edge that meets the square of half-size max_range * (1 + 2^-11) around the origin, whatever the
    origin's magnitude, and drops ordinary far edges"""
    for R in (1e-6, 0.5, 3.0):
        for o in ((0.0, 0.0), (1000.3, -17.25), (-3.7e5, 2.2e5)):
            d = _lib.TcLidarDesc(64, 360.0, R, 0.0, 0.0)
            cs = (math.cos(0.7), math.sin(0.7))
            h = R * (1 + 2.0 ** -11)
            for sx, sy in ((1, 0), (-1, 0), (0, 1), (0, -1)):
                # a short edge parallel to the side, just inside the grown square
                x, y = o[0] + sx * h, o[1] + sy * h
                a = (x - abs(sy) * 1e-3 * R, y - abs(sx) * 1e-3 * R)
                b = (x + abs(sy) * 1e-3 * R, y + abs(sx) * 1e-3 * R)
                assert host_keep(d, o, cs, a, b), (R, o, sx, sy)
            far = (o[0] + 10 * R + 1.0, o[1] + 10 * R + 1.0)
            assert not host_keep(d, o, cs, far, (far[0] + 0.1 * R, far[1] + 0.3 * R))


def cfg_with(lidar, map_name="simple_layout"):
    c = make_config(map_name, "classes")
    c["lidar"] = lidar
    return c


def test_lidar_params_defaults():
    assert lidar_params(make_config("knuffingen", "classes"), 5) is None
    assert lidar_params(cfg_with({}), 5) == {"rays": 64, "fov": 360.0, "max_range": 0.5, "origin": [0.0, 0.0], "classes": 5}
    p = lidar_params(cfg_with({"rays": 1024, "fov": 1e-3, "max_range": 1e6, "origin": [-0.1, 2]}), 3)
    assert p == {"rays": 1024, "fov": 1e-3, "max_range": 1e6, "origin": [-0.1, 2.0], "classes": 3}


@pytest.mark.parametrize("bad", [
    [], {"rays": 0}, {"rays": 1025}, {"rays": 64.0}, {"rays": True}, {"rays": "64"},
    {"fov": 0}, {"fov": -10}, {"fov": 360.5}, {"fov": float("nan")}, {"fov": "wide"},
    {"max_range": 0}, {"max_range": -1.0}, {"max_range": float("inf")}, {"max_range": float("nan")}, {"max_range": None},
    {"origin": [0.1]}, {"origin": [0.0, float("nan")]}, {"origin": [float("inf"), 0.0]}, {"origin": "front"}, {"origin": [True, 0.0]},
    {"range": 0.5},
])
def test_lidar_params_rejects(bad):
    with pytest.raises(ValueError):
        lidar_params(cfg_with(bad), 5)


@pytest.mark.parametrize("desc,what", [
    ((0, 360.0, 0.5, 0.0, 0.0), "rays"), ((1025, 360.0, 0.5, 0.0, 0.0), "rays"), ((64, 0.0, 0.5, 0.0, 0.0), "fov"),
    ((64, 360.0001, 0.5, 0.0, 0.0), "fov"), ((64, float("nan"), 0.5, 0.0, 0.0), "fov"), ((64, 90.0, 0.0, 0.0, 0.0), "max_range"),
    ((64, 90.0, float("inf"), 0.0, 0.0), "max_range"), ((64, 90.0, float("nan"), 0.0, 0.0), "max_range"),
    ((64, 90.0, 0.5, float("nan"), 0.0), "origin"), ((64, 90.0, 0.5, 0.0, float("-inf")), "origin"),
    ((64, 90.0, 0.5, 0.0, 0.0), "null handle"), ((1024, 360.0, 1e6, 1.0, -1.0), "null handle"),
])
def test_set_lidar_validates_before_any_device_call(desc, what):
    """tc_set_lidar checks the description before the handle (TC_ERR_INVALID and the rule that failed); a valid description then
    fails on the null handle. tc_render_lidar without a handle is TC_ERR_INVALID as well (TC_ERR_STATE, no scan set, needs a
    handle: tests/test_gpu_lidar.py)."""
    L = _lib.lib()
    d = _lib.TcLidarDesc(*desc)
    buf = (C.c_float * 4)()
    assert L.tc_set_lidar(None, C.byref(d), C.cast(buf, C.c_void_p)) == -1
    assert what in L.tc_last_error().decode()
    assert L.tc_set_lidar(None, None, C.cast(buf, C.c_void_p)) == -1 and b"null description" in L.tc_last_error()
    assert L.tc_set_lidar(None, None, None) == -1 and b"null handle" in L.tc_last_error()
    assert L.tc_render_lidar(None, None, None) == -1 and b"null handle" in L.tc_last_error()
