"""CPU checks of camera rigs (the config's `cameras` list, include/tinycarlo_b200.h tc_create_rig): the validation of
config.camera_rig, the per-view camera rows an env uploads, the view order of the poses in the host build of the tracking
step and the C ABI's argument checks, none of which needs a GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from rig_util import REAR, HostRig, oracle_pose
from tinycarlo_b200 import _lib
from tinycarlo_b200.camera_params import view_rows
from tinycarlo_b200.config import camera_rig, car_param_row, make_config, resolve_map_path
from tinycarlo_b200.maptables import MapTables

pytest.importorskip("cv2")


def cfg_with(cameras):
    cfg = make_config("knuffingen", "classes")
    cfg["cameras"] = cameras
    return cfg


THREE = [{}, REAR, {"fov": 110, "max_range": 1.0, "line_thickness": 4, "position": [0.01, 0.0, 0.05]}]


def test_without_the_key_there_is_no_rig():
    assert camera_rig(make_config("knuffingen", "classes")) is None


@pytest.mark.parametrize("cameras", [[], {}, "front", ({},), [{}, "rear"], [{}, [22, 0, 180]], [None]])
def test_rig_must_be_a_non_empty_list_of_mappings(cameras):
    with pytest.raises(ValueError, match="cameras"):
        camera_rig(cfg_with(cameras))


@pytest.mark.parametrize("entry,what", [({"zoom": 2}, "unknown"), ({"fov": 90, "pitch": 3}, "unknown"),
                                        ({"resolution": [84, 84]}, "resolution"), ({"resolution": [128, 160]}, "resolution")])
def test_rig_rejects_unknown_keys_and_resolution(entry, what):
    with pytest.raises(ValueError, match=what):
        camera_rig(cfg_with([{}, entry]))


@pytest.mark.parametrize("max_range", [None, 0])
def test_rig_entry_max_range_checked(max_range):
    with pytest.raises(ValueError, match="max_range"):
        camera_rig(cfg_with([{}, {"max_range": max_range}]))


@pytest.mark.parametrize("t", [0, 256, 2.0, True])
def test_rig_entry_thickness_checked(t):
    with pytest.raises(ValueError, match="line_thickness"):
        camera_rig(cfg_with([{"line_thickness": t}]))


def test_rig_entries_override_the_camera_section():
    cfg = cfg_with(THREE)
    rig = camera_rig(cfg)
    cam = cfg["camera"]
    assert len(rig) == 3
    assert rig[0] == {**cam, "resolution": list(cam["resolution"])}
    assert rig[1]["orientation"] == [22, 0, 180] and rig[1]["fov"] == cam["fov"] and rig[1]["position"] == cam["position"]
    assert rig[2]["fov"] == 110 and rig[2]["max_range"] == 1.0 and rig[2]["line_thickness"] == 4
    assert all(r["resolution"] == cam["resolution"] for r in rig)
    assert len(camera_rig(cfg_with([{}]))) == 1


def test_rig_rows_are_the_oracle_matrices_env_major():
    """the rows a rig env uploads (view_rows, as TinyCarloVecEnv builds them): oracle.camera_matrices + pack_cam of each
    merged section, view v = env * M + m"""
    cfg = cfg_with(THREE)
    rig = camera_rig(cfg)
    n, M = 5, len(rig)
    rows, thick = view_rows(rig, n)
    assert rows.shape == (n * M, 20) and thick.shape == (n * M,) and thick.dtype == np.int32
    for m, c in enumerate(rig):
        E, K = orc.camera_matrices(c["position"], c["orientation"], c["fov"], c["resolution"])
        want = orc.pack_cam(E, K, c["max_range"])
        for i in range(n):
            assert np.array_equal(rows[i * M + m], want), (i, m)
            assert thick[i * M + m] == c["line_thickness"]
    # without a rig: the config's camera, one row per env, as before
    rows1, thick1 = view_rows([rig[0]], n)
    assert np.array_equal(rows1, rows[0::M]) and np.array_equal(thick1, thick[0::M])


@pytest.mark.parametrize("M", [1, 3])
def test_host_rig_poses_follow_the_view_order(M):
    """the host build of the tracking step writes pose row i*M+m = orc_camera_pose(camera row i*M+m, state of env i) for
    reset and step, and in reset mode the view mask mask[i] for every view of env i (also when the env is not selected)"""
    cfg = cfg_with(THREE[:M])
    rig = camera_rig(cfg)
    tables = MapTables(resolve_map_path(cfg["map"], None), cfg["map"]["pixel_per_meter"], cfg["map"].get("spawn_points"))
    n = 24
    rng = np.random.default_rng(M)
    rows, thick = view_rows(rig, n)
    rows[2 * M::M, 16] = rng.uniform(0.3, 2.0, n - 2)   # per-env reach of camera 0 so that rows differ env to env
    host = HostRig(tables, n, M, car_param_row(cfg["car"], 1 / 30), rows, thick, 128, 160)
    spawn = rng.choice(cfg["map"]["spawn_points"], n).astype(np.int32)

    def check(where):
        for i in range(n):
            for m in range(M):
                assert np.array_equal(host.pose[i * M + m], oracle_pose(rows[i * M + m], host.sf[i])), (where, i, m)
    host.reset(spawn, render=False)
    check("reset")
    assert (host.view_mask == 0xEE).all()   # no mask: no view mask written
    for t in range(6):
        cc = np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)], 1)   # reverse commands included
        host.step(cc, rng.integers(0, 4, n), render=False)
        check(f"step {t}")
    mask = (rng.random(n) < 0.5).astype(np.uint8)
    mask[:2] = [0, 1]
    before = host.pose.copy()
    host.reset(rng.choice(cfg["map"]["spawn_points"], n).astype(np.int32), mask=mask, render=False)
    assert np.array_equal(host.view_mask, np.repeat(mask, M))
    check("masked reset")
    keep = np.repeat(mask == 0, M)
    assert np.array_equal(host.pose[keep], before[keep])


def _desc():
    m = MapTables(resolve_map_path({"map_name": "knuffingen"}, None), 222, None)
    keep = [np.ascontiguousarray(a) for a in (m.ll_node_off, m.ll_edge_off, m.ll_nodes, m.ll_edges, m.colors, m.lp_nodes, m.lp_edges,
                                              m.lp_orient, m.lp_orient_rev)]
    desc = _lib.TcMapDesc(m.n_classes, *(k.ctypes.data for k in keep[:5]), len(m.lp_nodes), len(m.lp_edges), *(k.ctypes.data for k in keep[5:]))
    return desc, keep, m.n_classes


@pytest.mark.parametrize("n_envs,n_cameras,what", [(4, 0, "n_cameras"), (4, -1, "n_cameras"), (2**28, 4, "exceeds"), (2**30, 2, "exceeds")])
def test_create_rig_rejects_bad_camera_counts(n_envs, n_cameras, what):
    """checked before any CUDA call: n_cameras >= 1, and num_envs * n_cameras * C must fit the int block index of the
    per-class grid (Knuffingen has 5 classes)"""
    L = _lib.lib()
    desc, keep, C_ = _desc()
    assert n_cameras < 1 or n_envs * n_cameras * C_ > 2**31 - 1
    sim = _lib.TcSimDesc(128, 160, _lib.TC_OBS_CLASSES)
    h = C.c_void_p()
    assert L.tc_create_rig(C.byref(desc), C.byref(sim), n_envs, n_cameras, 0, C.byref(h)) == -1   # TC_ERR_INVALID
    assert what in L.tc_last_error().decode()
    assert not h
