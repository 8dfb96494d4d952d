"""CPU checks at the class-count and line-thickness edges that the bundled maps and the shipped configs never reach:
laneline layers without edges (in the oracle and in the host build of the kernel arithmetic), lines 9 to 255 pixels thick
against cv2.polylines, and the validation of the line thickness and of the class count."""
import numpy as np
import pytest

import map_shapes_util as M
from hosttest_util import HostCore, polyline
from oracle import oracle as orc
from tinycarlo_b200.camera_params import camera_row
from tinycarlo_b200.config import car_param_row, make_config
from tinycarlo_b200.maptables import MapTables

cv2 = pytest.importorskip("cv2")

EMPTY_AT, NODES_ONLY_AT = 2, 4   # class positions of the inserted layers (the five Knuffingen layers keep their order)


def _degenerate_knuffingen():
    d = M.knuffingen()
    extra = {EMPTY_AT: ("empty", {"layer_color": [1, 2, 3], "nodes": [], "edges": []}),
             NODES_ONLY_AT: ("nodes_only", {"layer_color": [4, 5, 6], "nodes": [list(p) for p in d["lanelines"]["hold"]["nodes"]], "edges": []})}
    return d, M.with_extra_layers(d, extra)


def _rollout(make_env, n, steps, seed):
    """reset + steps of random forward actions with random maneuvers; -> per step (info, nearest, frames, flags)"""
    rng = np.random.default_rng(seed)
    env = make_env()
    spawn = rng.choice(M.SPAWN_KNUFF, n).astype(np.int32)
    env.reset(spawn)
    out = [(env.info.copy(), env.nearest.copy(), env.obs.copy(), env.terminated.copy(), env.truncated.copy())]
    for _ in range(steps):
        cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
        man = rng.integers(0, 4, n).astype(np.int32)
        env.step(cc.astype(np.float64) if isinstance(env, orc.OracleVecEnv) else cc, man)
        out.append((env.info.copy(), env.nearest.copy(), env.obs.copy(), env.terminated.copy(), env.truncated.copy()))
    return out


@pytest.mark.parametrize("impl", ["oracle", "host"])
def test_laneline_layers_without_edges(impl):
    """A class with no nodes and a class with nodes but no edges: distance 0 and nearest edge -1 (the reference raises
    ValueError in min([]), layer.py:33-44; the device defines it so, tc_core.cuh tc_get_info), an empty plane, and the
    other classes exactly as on the map without those layers."""
    plain, extra = _degenerate_knuffingen()
    cfg = make_config("knuffingen", "classes", cam={"resolution": [64, 80]})
    cc = cfg["camera"]
    H, W = cc["resolution"]
    n, steps = 48, 12
    car = car_param_row(cfg["car"], 1 / 30)
    cam = camera_row(cc["position"], cc["orientation"], cc["fov"], cc["resolution"], cc["max_range"])

    def make(data):
        if impl == "oracle":
            return lambda: orc.OracleVecEnv(orc.OracleMap(data, M.PPM, M.SPAWN_KNUFF), n, car, cam, cc["line_thickness"], H, W)
        return lambda: HostCore(MapTables(data, M.PPM, M.SPAWN_KNUFF), n, car, cam, cc["line_thickness"], H, W)
    got, want = _rollout(make(extra), n, steps, 1), _rollout(make(plain), n, steps, 1)
    keep = [c for c in range(7) if c not in (EMPTY_AT, NODES_ONLY_AT)]
    tracked = 0
    for t, ((i_g, e_g, o_g, te_g, tr_g), (i_w, e_w, o_w, te_w, tr_w)) in enumerate(zip(got, want)):
        for c in (EMPTY_AT, NODES_ONLY_AT):
            assert (i_g[:, 4 + c] == 0).all() and (e_g[:, c] == -1).all(), (impl, t, c, i_g[:, 4 + c])
            assert not o_g[:, c].any(), (impl, t, c)
        assert np.array_equal(i_g[:, :4], i_w[:, :4]) and np.array_equal(i_g[:, 4:][:, keep], i_w[:, 4:]), (impl, t)
        assert np.array_equal(e_g[:, keep], e_w), (impl, t)
        assert np.array_equal(o_g[:, keep], o_w), (impl, t)
        assert np.array_equal(te_g, te_w) and np.array_equal(tr_g, tr_w), (impl, t)
        tracked += int((e_w >= 0).all(axis=1).sum())
    assert tracked > n * steps // 2, "too few steps with a tracked edge to say anything about the distances"


def test_oracle_and_host_agree_on_degenerate_layers():
    """The same rollout on the map with the extra layers through the oracle and through the host build of the kernels."""
    _, extra = _degenerate_knuffingen()
    cfg = make_config("knuffingen", "classes", cam={"resolution": [64, 80]})
    cc = cfg["camera"]
    H, W = cc["resolution"]
    n = 32
    car = car_param_row(cfg["car"], 1 / 30)
    cam = camera_row(cc["position"], cc["orientation"], cc["fov"], cc["resolution"], cc["max_range"])
    th = np.resize(np.array(M.THICKNESSES, np.int32), n)
    o = _rollout(lambda: orc.OracleVecEnv(orc.OracleMap(extra, M.PPM, M.SPAWN_KNUFF), n, car, cam, th, H, W), n, 10, 2)
    h = _rollout(lambda: HostCore(MapTables(extra, M.PPM, M.SPAWN_KNUFF), n, car, cam, th, H, W), n, 10, 2)
    for t, (a, b) in enumerate(zip(o, h)):
        np.testing.assert_allclose(b[0], a[0], rtol=1e-9, atol=1e-11, err_msg=f"info step {t}")
        for k in (1, 2, 3, 4):
            assert np.array_equal(a[k], b[k]), (t, k)


THICK = list(range(9, 65)) + [100, 200, 255]


@pytest.mark.parametrize("H,W", [(84, 84), (128, 160), (480, 640), (45, 71)])
def test_thick_lines_vs_cv2(H, W):
    """cv2.polylines with thicknesses 9..64, 100, 200 and 255 against the oracle's restatement and the host build of the
    kernels' rasteriser (both set-up variants), endpoints in the frame, near it and far away."""
    rng = np.random.default_rng(H * 1000 + W)
    bad = []
    for t in THICK:
        for k in range(10):
            def pt(kind):
                if kind == 0:
                    return int(rng.integers(0, W)), int(rng.integers(0, H))
                if kind == 1:
                    s = 3 * t + 50
                    return int(rng.integers(-s, W + s)), int(rng.integers(-s, H + s))
                return int(rng.integers(-10**6, 10**6)), int(rng.integers(-10**6, 10**6))
            p0, p1 = pt(k % 3), pt((k // 3) % 2)
            a = np.zeros((H, W), np.uint8)
            cv2.polylines(a, np.int32([[p0, p1]]), False, 255, t)
            b = np.zeros((H, W), np.uint8)
            orc.polyline(b, p0, p1, [255], t)
            if not np.array_equal(a, b):
                bad.append(("oracle", p0, p1, t))
            for nl in (32, -2):
                if not np.array_equal(a, polyline(H, W, p0, p1, t, nlanes=nl)):
                    bad.append((f"host nlanes={nl}", p0, p1, t))
    assert not bad, bad[:5]


@pytest.mark.parametrize("t", [0, -1, 2.5, True, 256, None, "3"])
def test_camera_line_thickness_is_validated(t):
    from tinycarlo_b200.config import camera_params
    with pytest.raises(ValueError, match="line_thickness"):
        camera_params({"max_range": 0.5, "line_thickness": t})


def test_camera_line_thickness_range_is_accepted():
    from tinycarlo_b200.config import camera_params
    assert camera_params({"max_range": 0.5})["line_thickness"] == 1
    for t in (1, 2, 255, np.int32(64)):
        assert camera_params({"max_range": 0.5, "line_thickness": t})["line_thickness"] == int(t)


def test_per_env_line_thickness_is_validated():
    """set_camera_params / set_camera_rows (and through them the grouped env) take per-env arrays: the same range."""
    torch = pytest.importorskip("torch")
    from tinycarlo_b200.vec_env import TinyCarloVecEnv
    rows = TinyCarloVecEnv._thickness_rows
    assert rows(np.array([1, 9, 255]), (3,)).tolist() == [1, 9, 255]
    assert rows(torch.tensor([2, 64], dtype=torch.int32), (2,)).dtype == np.int32
    assert rows(7, (4,)).tolist() == [7] * 4
    for v in ([0, 1], [1, 256], [-1], [2.5, 3.0], np.array([True, True]), np.array([3.0])):
        with pytest.raises(ValueError, match="line_thickness"):
            rows(v, (len(np.atleast_1d(v)),))


def test_class_count_is_validated():
    d = M.knuffingen()
    layers = list(d["lanelines"].values())

    def with_n(n):
        e = dict(d)
        e["lanelines"] = {f"c{i}": layers[i % len(layers)] for i in range(n)}
        return e
    assert MapTables(with_n(16), M.PPM, M.SPAWN_KNUFF).n_classes == 16
    assert MapTables(M.k16(), M.PPM, M.SPAWN_KNUFF).n_classes == 16
    with pytest.raises(ValueError, match="17 laneline layers"):
        MapTables(with_n(17), M.PPM, M.SPAWN_KNUFF)
