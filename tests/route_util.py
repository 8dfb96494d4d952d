"""numpy restatement of the navigation goals' contract (include/tinycarlo_b200.h TcRouteDesc): the edge transitions with
tc_pick_edge's self-loop quirk, the route table by Bellman-Ford (an independent route to the fixed point the library reaches
with Dijkstra), the per-env update, and goal draws on plain numpy Generators. Also the host build's entry points and small
synthetic lanepath maps."""
import ctypes as C
import json
import math
import os

import numpy as np

from hosttest_util import HostCore, P, ht
from tinycarlo_b200.maptables import MapTables

MANEUVERS = (0, 1, 3)


def clip_angle(a):
    if not abs(a) <= 1.0e4:
        return math.nan
    while a > math.pi:
        a -= 2 * math.pi
    while a < -math.pi:
        a += 2 * math.pi
    return a


def pick_next(t: MapTables, node, orientation):
    """tc_pick_edge over the edges leaving `node` (edge-list order): a single edge is returned as it is; otherwise the
    self-loops are dropped from the orientation list, and the winner's position indexes the UNfiltered list"""
    cand = [int(e) for e in np.nonzero(t.lp_edges[:, 0] == node)[0]]
    if not cand:
        return -1
    if len(cand) == 1:
        return cand[0]
    best, bd, k = -1, 0.0, 0
    for e in cand:
        if t.lp_edges[e, 1] == node:
            continue
        d = abs(clip_angle(float(t.lp_orient[e]) - orientation))
        if best < 0 or d < bd:
            best, bd = k, d
        k += 1
    return -1 if best < 0 else cand[best]


def transitions(t: MapTables):
    """T [Q, 3]: the edge after e under m = 0, 1, 3 (-1: none)"""
    Q = len(t.lp_edges)
    T = np.full((Q, 3), -1, np.int64)
    for e in range(Q):
        for j, m in enumerate(MANEUVERS):
            T[e, j] = pick_next(t, int(t.lp_edges[e, 1]), clip_angle(float(t.lp_orient[e]) + m * math.pi / 2))
    return T


def edge_lengths(t: MapTables):
    a, b = t.lp_nodes[t.lp_edges[:, 0]], t.lp_nodes[t.lp_edges[:, 1]]
    return np.sqrt((a[:, 0] - b[:, 0]) * (a[:, 0] - b[:, 0]) + (a[:, 1] - b[:, 1]) * (a[:, 1] - b[:, 1]))


def route_table(t: MapTables, goals):
    """(D float64 [G, Q], cmd int8 [G, Q]) by Bellman-Ford from +inf: the least fixed point of the contract's equations"""
    goals = np.asarray(goals, np.int64)
    T, L = transitions(t), edge_lengths(t)
    term = t.lp_edges[None, :, 1] == goals[:, None]
    D = np.where(term, 0.0, np.inf)

    def candidates(D):
        c = np.full(D.shape + (3,), np.inf)
        for j in range(3):
            ok = T[:, j] >= 0
            c[:, ok, j] = L[T[ok, j]][None, :] + D[:, T[ok, j]]
        return c
    while True:
        nd = np.where(term, 0.0, candidates(D).min(axis=2))
        if np.array_equal(nd, D):
            break
        D = nd
    c = candidates(D)
    cmd = np.full(D.shape, -1, np.int8)
    live = (D != 0) & np.isfinite(D)
    for j in (2, 1, 0):   # the smallest m attaining the minimum wins: written last
        hit = live & (c[:, :, j] == D)
        cmd[hit] = MANEUVERS[j]
    return D, cmd


def route_edge(t: MapTables, si):
    pe, pn0, pn1 = int(si[10]), int(si[2]), int(si[3])
    if si[0] <= 0 or pe < 0 or pe >= len(t.lp_edges) or pn0 < 0 or pn1 < 0 or pn1 >= len(t.lp_nodes):
        return -1
    return pe


def tdist(ax, ay, bx, by):
    dx, dy = ax - bx, ay - by
    return math.sqrt(dx * dx + dy * dy)


def evaluate(t, D, cmd, goals, reach, pe, pn1, fx, fy, k):
    """-> (command, distance, reached) of goal index k"""
    if k < 0 or pe < 0 or not D[k, pe] < math.inf:
        return -1, math.inf, False
    d = tdist(fx, fy, float(t.lp_nodes[pn1, 0]), float(t.lp_nodes[pn1, 1]))
    return int(cmd[k, pe]), d + float(D[k, pe]), bool(pn1 == goals[k] and d <= reach)


def draw(t, D, goals, reach, pe, pn1, fx, fy, gen):
    if pe < 0:
        return -1
    at_pn1 = tdist(fx, fy, float(t.lp_nodes[pn1, 0]), float(t.lp_nodes[pn1, 1])) <= reach
    valid = [k for k in range(len(goals)) if D[k, pe] < math.inf and not (at_pn1 and goals[k] == pn1)]
    if not valid:
        return -1
    return valid[int(gen.integers(0, len(valid)))]


def update(t, D, cmd, goals, reach, on_reach, mode, sf, si, gens, k, prev, mask=None, was_reset=None):
    """The contract for every env (mode 0 after a step, 1 draw, 2 recompute; masks apply to modes 1 and 2). gens: one numpy
    Generator per env (the goal streams), advanced in place; k, prev: updated in place. -> dict of the outputs [N] (None for
    envs left alone) and the terminate flags"""
    n = len(sf)
    out = {key: [None] * n for key in ("goal", "gx", "gy", "command", "distance", "progress", "reached", "terminate")}
    for i in range(n):
        if mode != 0 and mask is not None and not mask[i]:
            continue
        pe, pn1 = route_edge(t, si[i]), int(si[i, 3])
        fx, fy = float(sf[i, 5]), float(sf[i, 6])
        ki = int(k[i]) if 0 <= k[i] < len(goals) else -1
        progress, reached, terminate = 0.0, False, False
        do_draw = mode == 1 or (mode == 0 and was_reset is not None and bool(was_reset[i]))
        if not do_draw:
            c, dist, reached = evaluate(t, D, cmd, goals, reach, pe, pn1, fx, fy, ki)
            if mode == 0:
                if math.isfinite(prev[i]) and math.isfinite(dist):
                    progress = float(prev[i]) - dist
                if reached:
                    if on_reach == 1:
                        terminate = True
                    else:
                        do_draw = True
        if do_draw:
            ki = draw(t, D, goals, reach, pe, pn1, fx, fy, gens[i])
            c, dist, _ = evaluate(t, D, cmd, goals, reach, pe, pn1, fx, fy, ki)
        k[i], prev[i] = ki, dist
        node = int(goals[ki]) if ki >= 0 else -1
        out["goal"][i] = node
        out["gx"][i] = np.float32(t.lp_nodes[node, 0]) if node >= 0 else np.float32(np.nan)
        out["gy"][i] = np.float32(t.lp_nodes[node, 1]) if node >= 0 else np.float32(np.nan)
        out["command"][i], out["distance"][i], out["progress"][i] = c, np.float32(dist), np.float32(progress)
        out["reached"][i], out["terminate"][i] = reached, terminate
    return out


def generators(seeds):
    """the goal stream of every env as numpy defines it: Generator(PCG64(SeedSequence(seed).spawn(1)[0]))"""
    return [np.random.Generator(np.random.PCG64(np.random.SeedSequence(int(s)).spawn(1)[0])) for s in seeds]


def generator_rows(gens):
    """uint64 [N, 5] TC_RNG_* rows of numpy Generators"""
    rows = np.zeros((len(gens), 5), np.uint64)
    for i, g in enumerate(gens):
        st = g.bit_generator.state
        s, inc = st["state"]["state"], st["state"]["inc"]
        buf = ((1 << 32) | st["uinteger"]) if st["has_uint32"] else 0
        rows[i] = [s >> 64, s & (2**64 - 1), inc >> 64, inc & (2**64 - 1), buf]
    return rows


# ------------------------------------------------------------------------------------------------ host build
def _bind():
    L = ht()
    if not getattr(L, "_route_bound", False):
        vp = C.c_void_p
        L.ht_route_table.argtypes = [vp, C.c_int, vp, vp, vp]
        L.ht_route_update.argtypes = [vp, C.c_int, vp, vp, vp, C.c_double, C.c_int, C.c_int, C.c_int] + [vp] * 15
        L._route_bound = True
    return L


def host_map(t: MapTables):
    """a host-build map of the tables (HostCore with no envs to speak of)"""
    return HostCore(t, 1, np.zeros(8), np.zeros(20), 1, 8, 8)


def host_table(hm, goals, Q):
    goals = np.ascontiguousarray(goals, np.int32)
    D = np.zeros((len(goals), Q))
    cmd = np.zeros((len(goals), Q), np.int8)
    _bind().ht_route_table(hm.h, len(goals), P(goals), P(D), P(cmd))
    return D, cmd


def host_update(hm, goals, D, cmd, reach, on_reach, mode, sf, si, rng, k, prev, mask=None, was_reset=None, terminated=None, done=None):
    """ht_route_update; rng, k, prev, terminated, done are updated in place -> dict of the outputs"""
    n = len(sf)
    goals = np.ascontiguousarray(goals, np.int32)
    o = {"goal": np.full(n, -7, np.int32), "goal_position": np.full((n, 2), -7, np.float32), "command": np.full(n, -7, np.int32),
         "distance": np.full(n, -7, np.float32), "progress": np.full(n, -7, np.float32), "reached": np.full(n, 7, np.uint8)}
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    w = None if was_reset is None else np.ascontiguousarray(was_reset, np.uint8)
    _bind().ht_route_update(hm.h, len(goals), P(goals), P(np.ascontiguousarray(D)), P(np.ascontiguousarray(cmd)), float(reach), int(on_reach), n,
                            int(mode), P(np.ascontiguousarray(sf, np.float64)), P(np.ascontiguousarray(si, np.int32)), P(m), P(w), P(rng), P(k),
                            P(prev), P(o["goal"]), P(o["goal_position"]), P(o["command"]), P(o["distance"]), P(o["progress"]),
                            P(o["reached"]), P(terminated), P(done))
    return o


def assert_outputs_equal(got, want, envs=None, what=""):
    """host or device outputs (numpy) against update()'s, float32 bit patterns"""
    n = len(want["goal"])
    for i in (range(n) if envs is None else envs):
        if want["goal"][i] is None:
            continue
        exp = [want["goal"][i], want["command"][i], bool(want["reached"][i])]
        act = [int(got["goal"][i]), int(got["command"][i]), bool(got["reached"][i])]
        assert act == exp, f"{what} env {i}: goal/command/reached {act} != {exp}"
        for key, w in (("distance", want["distance"][i]), ("progress", want["progress"][i]))+ \
                (("gx", want["gx"][i]), ("gy", want["gy"][i])):
            g = got["goal_position"][i, 0 if key == "gx" else 1] if key in ("gx", "gy") else got[key][i]
            assert np.float32(g).view(np.int32) == np.float32(w).view(np.int32) or (np.isnan(g) and np.isnan(w)), \
                f"{what} env {i}: {key} {g!r} != {w!r}"


# ------------------------------------------------------------------------------------------------ synthetic maps
def write_map(directory, name, nodes, edges):
    """a map JSON (pixel_per_meter 1) with the given lanepath and one small laneline layer"""
    data = {"width": 100, "height": 100,
            "lanelines": {"solid": {"layer_color": [255, 255, 255], "nodes": [[0, -5], [1, -5]], "edges": [[0, 1]]}},
            "lanepath": {"layer_color": [0, 0, 255], "nodes": [list(map(float, p)) for p in nodes], "edges": [list(e) for e in edges]}}
    path = os.path.join(str(directory), name + ".json")
    with open(path, "w") as f:
        json.dump(data, f)
    return path


# A(0) -> B(1); B has three successors: straight to the dead end S(2), right to R(3), left to Lf(4); R and Lf both lead to
# G(5) over equally long edges, so the route from (A, B) ties between m = 1 and m = 3. G -> H(6) is a dead end; K(9) -> I(7) ->
# J(8) is a chain no edge leads into, so I and J are goals no car on the rest of the map can reach.
JUNCTION = ([[0, 0], [1, 0], [2, 0], [2, 1], [2, -1], [3, 0], [4, 0], [5, 0], [6, 0]],
            [[0, 1], [1, 2], [1, 3], [1, 4], [3, 5], [4, 5], [5, 6], [9, 7], [7, 8]])
# W(0) -> X(1); X's edges in list order: a self-loop, X -> Y(2) straight ahead, X -> Z(3) to the right. The straight pick wins
# position 0 of the filtered list and so returns the self-loop; the right pick returns X -> Y. Y and Z continue to V(4), U(5).
SELF_LOOP = ([[0, 0], [1, 0], [2, 0], [1, 1], [3, 0], [1, 2]],
             [[0, 1], [1, 1], [1, 2], [1, 3], [2, 4], [3, 5]])
SYNTHETIC = {"junction": JUNCTION, "self_loop": SELF_LOOP}


def synthetic_tables(directory, name):
    nodes, edges = SYNTHETIC[name]
    if name == "junction":
        nodes = nodes + [[5, 1]]   # node 9: start of the edge nothing reaches
    return MapTables(write_map(directory, name, nodes, edges), 1)
