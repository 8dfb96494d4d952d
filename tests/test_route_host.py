"""CPU checks of the navigation goals: the host build of the route table (tc_route.h) and of the per-env update (tc_core.cuh,
what tc_route_kernel runs) against the numpy restatement of the contract in tests/route_util.py, bit for bit; the goal
streams against numpy's SeedSequence.spawn; the validation of the config's `navigation` section and of the C entry points."""
import ctypes as C
import math

import numpy as np
import pytest

import route_util as R
from hosttest_util import HostCore
from tinycarlo_b200 import _lib
from tinycarlo_b200.config import CAR_SHIPPED, MAPS_DIR, PPM, SPAWN_KNUFF, car_param_row, make_config, navigation_params
from tinycarlo_b200.pcg64 import VecPCG64
from tinycarlo_b200.spawn import goal_stream_states, spawn_stream_states, stream_seeds
from tinycarlo_b200.maptables import MapTables

MAPS = ["knuffingen", "simple_layout", "formula_student_track", "formula_student_skidpad"]


def bundled(name):
    return MapTables(f"{MAPS_DIR}/{name}.json", PPM[name], SPAWN_KNUFF if name == "knuffingen" else None)


def every_node_with_predecessor(t):
    return sorted({int(v) for v in t.lp_edges[:, 1]})


def check_table(t, goals):
    hm = R.host_map(t)
    D, cmd = R.host_table(hm, goals, len(t.lp_edges))
    Do, co = R.route_table(t, goals)
    assert np.array_equal(D.view(np.int64), Do.view(np.int64)), "route distances differ from the oracle"
    assert np.array_equal(cmd, co), "route commands differ from the oracle"
    return D, cmd


@pytest.mark.parametrize("name", MAPS)
def test_route_table_bundled_maps(name):
    t = bundled(name)
    D, cmd = check_table(t, every_node_with_predecessor(t))
    assert np.isfinite(D).any() and (cmd >= 0).any()
    assert set(np.unique(cmd)) <= {-1, 0, 1, 3}


def test_knuffingen_routes_between_spawn_points():
    """the issue's numbers: 99 of the 420 ordered pairs of distinct spawn points have no route"""
    t = bundled("knuffingen")
    D, _ = R.route_table(t, SPAWN_KNUFF)
    first = [int(np.nonzero(t.lp_edges[:, 0] == s)[0][0]) for s in SPAWN_KNUFF]   # the spawn pose's edge (tc_car_reset)
    none = sum(1 for a, ea in zip(SPAWN_KNUFF, first) for k, b in enumerate(SPAWN_KNUFF) if a != b and not np.isfinite(D[k, ea]))
    assert none == 99


@pytest.mark.parametrize("name", ["junction", "self_loop"])
def test_route_table_synthetic(name, tmp_path):
    t = R.synthetic_tables(tmp_path, name)
    check_table(t, every_node_with_predecessor(t))


def test_junction_ties_break_in_maneuver_order(tmp_path):
    """equal-length routes right and left of the dead end straight ahead: the command is 1 (0, 1, 3 order), not 3"""
    t = R.synthetic_tables(tmp_path, "junction")
    goals = every_node_with_predecessor(t)
    D, cmd = check_table(t, goals)
    T = R.transitions(t)
    e_ab, k_g = 0, goals.index(5)
    assert [int(v) for v in T[e_ab]] == [1, 2, 3]   # straight: the dead end; right: B -> R; left: B -> Lf
    assert cmd[k_g, e_ab] == 1 and D[k_g, e_ab] == math.sqrt(2) + math.sqrt(2)
    # the dead end and the chain nothing leads into
    assert not np.isfinite(D[goals.index(5), 1]) and (cmd[goals.index(5), 1] == -1)
    for g in (7, 8):
        reach = np.isfinite(D[goals.index(g)])
        assert set(np.nonzero(reach)[0]) <= {7, 8}


def test_self_loop_quirk(tmp_path):
    """the straight and left picks at X return the self-loop (the unfiltered list indexed), the right pick returns X -> Y, and
    no maneuver reaches Z"""
    t = R.synthetic_tables(tmp_path, "self_loop")
    goals = every_node_with_predecessor(t)
    D, cmd = check_table(t, goals)
    T = R.transitions(t)
    assert [int(v) for v in T[0]] == [1, 2, 1]   # W -> X: m = 0 and 3 the self-loop, m = 1 X -> Y
    assert cmd[goals.index(2), 0] == 0 and D[goals.index(2), 0] == 1.0   # to Y over the zero-length self-loop ties with m = 1
    assert not np.isfinite(D[goals.index(3), 0])   # Z: no maneuver picks X -> Z


# ------------------------------------------------------------------------------------------------ per-env update
def rollout_states(t, n, steps, rng):
    """states of a host rollout (reset at the spawn points, random actions), recorded after every step"""
    car = car_param_row(dict(CAR_SHIPPED, max_velocity=0.5), 1 / 30)
    hc = HostCore(t, n, car, np.zeros(20), 1, 8, 8)
    spawns = t.spawn_points or [int(v) for v in np.nonzero(t.has_successor)[0]]
    hc.reset(rng.choice(spawns, n).astype(np.int32), render=False)
    states = [(hc.sf.copy(), hc.si.copy())]
    for _ in range(steps):
        cc = np.stack([rng.uniform(0.3, 1.0, n), rng.uniform(-0.4, 0.4, n)], 1)
        hc.step(cc, rng.choice([0, 1, 3], n), render=False)
        states.append((hc.sf.copy(), hc.si.copy()))
    return states


def placed_states(t, goals, reach, rng):
    """states placed on purpose: the front axle on the goal node at the end of the tracked edge, just outside the radius, on
    a goal node that is the START of the tracked edge (pn0: must not count), no tracked edge, NaN"""
    rows = []
    for g in goals[:6]:
        e_in = int(np.nonzero(t.lp_edges[:, 1] == g)[0][0])
        n0 = int(t.lp_edges[e_in, 0])
        for off in (0.0, reach * 0.5, reach * 1.5):
            sf, si = np.zeros(8), np.full(16, -1, np.int32)
            si[0], si[1], si[2], si[3], si[10] = 1, 0, n0, g, e_in
            sf[5:7] = t.lp_nodes[g] + [off, 0.0]
            rows.append((sf, si))
        e_out = np.nonzero(t.lp_edges[:, 0] == g)[0]
        if len(e_out):
            sf, si = np.zeros(8), np.full(16, -1, np.int32)
            e = int(e_out[0])
            si[0], si[1], si[2], si[3], si[10] = 1, 0, g, int(t.lp_edges[e, 1]), e
            sf[5:7] = t.lp_nodes[g]
            rows.append((sf, si))
    sf, si = np.zeros(8), np.full(16, -1, np.int32)
    si[0] = 0
    rows.append((sf, si))
    sf, si = np.full(8, np.nan), rows[0][1].copy()
    rows.append((sf, si))
    return np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows])


def run_both(t, goals, reach, on_reach, frames, seeds, rng, modes):
    """ht_route_update and the oracle over the same frames -> number of draws, reaches"""
    hm = R.host_map(t)
    D, cmd = R.host_table(hm, goals, len(t.lp_edges))
    n = len(seeds)
    rows = goal_stream_states(n, None, seeds=np.asarray(seeds, np.uint64))
    gens = R.generators(seeds)
    k_h, p_h = np.full(n, -1, np.int32), np.full(n, np.inf)
    k_o, p_o = np.full(n, -1, np.int64), np.full(n, np.inf)
    draws = reaches = 0
    for f, ((sf, si), mode) in enumerate(zip(frames, modes)):
        mask = rng.random(n) < 0.6 if mode != 0 else None
        was = (rng.random(n) < 0.1) if mode == 0 else None
        term, done = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        got = R.host_update(hm, goals, D, cmd, reach, on_reach, mode, sf, si, rows, k_h, p_h, mask=mask, was_reset=was, terminated=term, done=done)
        want = R.update(t, D, cmd, goals, reach, on_reach, mode, sf, si, gens, k_o, p_o, mask=mask, was_reset=was)
        R.assert_outputs_equal(got, want, what=f"frame {f} mode {mode}")
        assert np.array_equal(k_h, k_o) and np.array_equal(p_h.view(np.int64), p_o.view(np.int64))
        assert np.array_equal(rows, R.generator_rows(gens)), "goal streams moved differently"
        exp_term = np.array([bool(v) for v in want["terminate"]], np.uint8)
        assert np.array_equal(term, exp_term) and np.array_equal(done, exp_term)
        reaches += sum(bool(v) for v in want["reached"] if v is not None)
        draws += int(mode == 1) * int((mask if mask is not None else np.ones(n, bool)).sum())
    return draws, reaches


@pytest.mark.parametrize("on_reach", [0, 1])
@pytest.mark.parametrize("name", ["knuffingen", "simple_layout"])
def test_update_over_recorded_states(name, on_reach):
    rng = np.random.default_rng(11 + on_reach)
    t = MapTables(f"{MAPS_DIR}/{name}.json", PPM[name], make_config(name, "classes")["map"].get("spawn_points"))
    goals = list(t.spawn_points)
    n = 64
    states = rollout_states(t, n, 60, rng)
    modes = [1] + [0] * 60
    modes[20] = 2
    draws, _ = run_both(t, goals, 0.05, on_reach, states, [7 + i for i in range(n)], rng, modes)
    assert draws > 0


@pytest.mark.parametrize("on_reach", [0, 1])
def test_update_over_placed_states(on_reach):
    """reaches (on the goal node, inside and outside the radius), the goal at pn0, no tracked edge, NaN; every mode"""
    rng = np.random.default_rng(5)
    t = bundled("knuffingen")
    goals = list(SPAWN_KNUFF)
    sf, si = placed_states(t, goals, 0.05, rng)
    n = len(sf)
    hm = R.host_map(t)
    D, cmd = R.host_table(hm, goals, len(t.lp_edges))
    # aim every env at the goal of its placement, then step at the same pose: reached where the front axle is within the radius
    k0 = np.array([goals.index(int(s[3])) if int(s[3]) in goals else 0 for s in si])
    seeds = np.arange(n) + 2**33
    rows = goal_stream_states(n, None, seeds=seeds.astype(np.uint64))
    gens = R.generators(seeds)
    k_h, p_h = k0.astype(np.int32), np.full(n, np.inf)
    k_o, p_o = k0.astype(np.int64), np.full(n, np.inf)
    reached_any = False
    for mode in (2, 0, 0, 1, 0):
        term, done = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        got = R.host_update(hm, goals, D, cmd, 0.05, on_reach, mode, sf, si, rows, k_h, p_h, terminated=term, done=done)
        want = R.update(t, D, cmd, goals, 0.05, on_reach, mode, sf, si, gens, k_o, p_o)
        R.assert_outputs_equal(got, want, what=f"mode {mode}")
        assert np.array_equal(rows, R.generator_rows(gens))
        assert np.array_equal(term, np.array(want["terminate"], np.uint8))
        reached_any |= bool(got["reached"].any())
        if mode == 0 and on_reach == 1:
            assert np.array_equal(term.astype(bool), got["reached"].astype(bool))
    assert reached_any
    # the goal at pn0 (the last placement of each goal) never counts; no tracked edge and NaN give +inf / NaN and no goal draw
    assert got["goal"][-2] == -1 and got["distance"][-2] == np.inf and got["command"][-2] == -1


def test_exhausted_draw_leaves_the_stream_alone(tmp_path):
    """an env whose tracked edge leads to no goal: goal -1, distance +inf, command -1, and its goal stream does not move"""
    t = R.synthetic_tables(tmp_path, "junction")
    goals = [8]   # reachable only from the chain no edge leads into
    hm = R.host_map(t)
    D, cmd = R.host_table(hm, goals, len(t.lp_edges))
    sf, si = np.zeros((1, 8)), np.full((1, 16), -1, np.int32)
    si[0, :4], si[0, 10] = [1, 0, 0, 1], 0
    rows = goal_stream_states(1, 3)
    before = rows.copy()
    k, p = np.full(1, -1, np.int32), np.full(1, np.inf)
    got = R.host_update(hm, goals, D, cmd, 0.05, 0, 1, sf, si, rows, k, p)
    assert got["goal"][0] == -1 and got["distance"][0] == np.inf and got["command"][0] == -1 and np.isnan(got["goal_position"][0]).all()
    assert np.array_equal(rows, before)
    # one valid goal: a draw of one candidate returns it without moving the stream either (numpy's integers(0, 1))
    goals = [5, 8]
    D, cmd = R.host_table(hm, goals, len(t.lp_edges))
    got = R.host_update(hm, goals, D, cmd, 0.05, 0, 1, sf, si, rows, k, p)
    assert got["goal"][0] == 5 and got["command"][0] == 1 and np.array_equal(rows, before)


# ------------------------------------------------------------------------------------------------ streams
def test_goal_streams_match_numpy_spawn():
    seeds = np.concatenate([np.arange(2000, dtype=np.uint64), np.arange(1000, dtype=np.uint64) + np.uint64(2**32 - 500),
                            np.array([2**63, 2**64 - 1], np.uint64)])
    rows = goal_stream_states(len(seeds), None, seeds=seeds)
    assert np.array_equal(rows, R.generator_rows(R.generators(seeds)))
    v = VecPCG64()
    v.load_device_rows(rows)
    gens = R.generators(seeds)
    for high in (3, 21, 1000003):
        assert np.array_equal(v.bounded(high), [g.integers(0, high) for g in gens])
    # offsets and the spawn streams, which stay numpy's SeedSequence(seed + offset + i)
    assert np.array_equal(goal_stream_states(50, 9, 100), R.generator_rows(R.generators(np.arange(50) + 109)))
    spawn = [np.random.Generator(np.random.PCG64(np.random.SeedSequence(int(s)))) for s in np.arange(50) + 109]
    assert np.array_equal(spawn_stream_states(50, 9, 100), R.generator_rows(spawn))
    assert stream_seeds(4, None).dtype == np.uint64


# ------------------------------------------------------------------------------------------------ validation
def test_navigation_params():
    t = bundled("knuffingen")
    cfg = make_config("knuffingen", "classes")
    assert navigation_params(cfg, t) is None
    cfg["navigation"] = {}
    p = navigation_params(cfg, t)
    assert p == {"goals": list(SPAWN_KNUFF), "reach_radius": 0.05, "on_reach": "resample"}
    t2 = MapTables(f"{MAPS_DIR}/knuffingen.json", PPM["knuffingen"])
    assert navigation_params(cfg, t2)["goals"] == every_node_with_predecessor(t2)
    cfg["navigation"] = {"goals": [2, 18], "reach_radius": 0, "on_reach": "terminate"}
    assert navigation_params(cfg, t)["on_reach"] == "terminate"
    no_pred = [i for i in range(len(t.lp_nodes)) if i not in set(every_node_with_predecessor(t))]
    bad = [[], "x", {"goals": []}, {"goals": [-1]}, {"goals": [len(t.lp_nodes)]}, {"goals": [1.0]}, {"goals": [True]},
           {"goals": list(range(4097))}, {"reach_radius": -0.1}, {"reach_radius": math.nan}, {"reach_radius": math.inf},
           {"reach_radius": "1"}, {"on_reach": "stop"}, {"route": 1}]
    if no_pred:
        bad.append({"goals": [no_pred[0]]})
    for nav in bad:
        cfg["navigation"] = nav
        with pytest.raises(ValueError):
            navigation_params(cfg, t)


def test_set_route_checks_the_description_without_a_device():
    L = _lib.lib()
    goals = np.array([1, 2], np.int32)

    def call(n=2, g=goals.ctypes.data, reach=0.05, on=0):
        d = _lib.TcRouteDesc(n, g, reach, on)
        rc = L.tc_set_route(None, C.byref(d), None, None, None, None)
        return rc, L.tc_last_error().decode()
    for kw, msg in (({"n": 0}, "n_goals"), ({"n": 4097}, "n_goals"), ({"g": None}, "goal list"), ({"reach": -1.0}, "reach_radius"),
                    ({"reach": math.nan}, "reach_radius"), ({"reach": math.inf}, "reach_radius"), ({"on": 2}, "on_reach")):
        rc, err = call(**kw)
        assert rc == -1 and msg in err, (kw, err)
    rc, err = call()
    assert rc == -1 and "null handle" in err
    assert L.tc_set_route(None, None, None, None, None, None) == -1 and "null handle" in L.tc_last_error().decode()
    assert L.tc_update_route(None, None, 1, None) == -1 and "null handle" in L.tc_last_error().decode()
