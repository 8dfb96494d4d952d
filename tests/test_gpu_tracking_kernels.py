"""The three tracking kernels at the env counts that select them (run with -m gpu on a B200).

A step runs one of three tracking kernels, and tc_create picks it from the env count alone (tc_api.cu): a warp per env
(tc_track_kernel<32>), 8 lanes per env (tc_track_kernel<8>) or a thread per env (tc_track_thread_kernel, the headline size).
The only way to run a kernel is a handle with that many envs, so every case here builds one at a count taken from the
rule (tracking_kernel) and checks the handle's choice first: if the rule changes, these cases fail instead of quietly
testing another kernel. The counts sit at the boundaries of the rule and leave the last block of each kernel partly
filled (the thread kernel's idle lanes shadow the last env inside the warp scans and must store nothing).

- test_tracking_kernel_matches_oracle: a rollout that reaches the rare paths of tracking (u-turn scans started by many
  lanes of a warp at once, cars placed inside / just outside / on the lines of / far beyond the nearest-laneline grid, NaN
  actions, next-step autoreset with device spawn draws, masked resets, mark_done + reset_done) against the CPU oracle.
- test_uturn_without_edge_truncates: a u-turn with no lanepath edge within +-30 degrees (DESIGN.md section 2).
- test_tracking_kernels_are_bit_identical: the same scenario through all three kernels, replica for replica, torch.equal.
- test_rig_on_the_larger_batch_kernels: a camera rig (M = 2) on <8> and the thread kernel, with a masked reset."""
import json
import os
import zlib

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from pair_util import PPM, make_config, oracle_env
from rig_util import REAR

pytestmark = pytest.mark.gpu

RTOL32 = 1e-5   # as test_gpu_parity: the north-star tolerance on the fp32 outputs
RTOL64 = 1e-9   # the float64 state and info
RES = [64, 96]  # small frames: the oracle renders them cheaply at 16k envs
T = 24          # steps of the scenario
SPAWN_TABLE = 32
DEAD_END = 92   # a Knuffingen lanepath node without successor: a reset on it fails
FOUR_BLOCK = {32: 8, 8: 32, 1: 128}   # envs per block of tc_track_kernel<32>, <8> and tc_track_thread_kernel


# ------------------------------------------------------------------------------------------------ which kernel, which counts
def tracking_kernel(n, sms):
    """(track_per_thread, lanes per env) that tc_create chooses for n envs on a device with `sms` SMs: a thread per env once
    8 lanes per env would need more than one wave of 3 blocks x 8 warps per SM, else 8 lanes per env once a warp per env
    would, else a warp per env (integer arithmetic, as in tc_api.cu)."""
    if n // 4 > 3 * 8 * sms:
        return 1, 1
    return 0, 8 if n > 3 * 8 * sms // 2 else 32


def kernel_counts(sms):
    """id -> env count at the boundaries of the rule, with partial last blocks (1771 / 1776 / 1777 / 14211 / 14212 / 16411 on
    a B200's 148 SMs)"""
    last32 = 12 * sms                    # largest count of the warp-per-env kernel
    last8 = 4 * (24 * sms) + 3           # largest count of the 8-lane kernel
    big = max(16384, last8 + 1)
    c = {"warp_partial": last32 - (last32 - 3) % 8,   # last 8-env block holds 3 envs
         "warp_last": last32,
         "group8_first": last32 + 1,
         "group8_last": last8,
         "thread_first": last8 + 1,
         "thread_big": big + (27 - big % 32) % 32}    # >= 16384, the last warp holds 27 envs
    return c


KERNEL_OF = {"warp_partial": (0, 32), "warp_last": (0, 32), "group8_first": (0, 8), "group8_last": (0, 8),
             "thread_first": (1, 1), "thread_big": (1, 1)}


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _count(case):
    n = kernel_counts(_sms())[case]
    assert tracking_kernel(n, _sms()) == KERNEL_OF[case], (case, n)
    return n


def _kernel_name(ri):
    return "tc_track_thread_kernel" if ri["track_per_thread"] else f"tc_track_kernel<{ri['track_lanes_per_env']}>"


def _vec(cfg, n, **kw):
    from tinycarlo_b200 import TinyCarloVecEnv
    return TinyCarloVecEnv(cfg, n, device="cuda:0", **kw)


_RENDER_KEYS = ("block_per_env", "envs_per_block", "prim_chunks", "render_smem", "banded_smem")
_RENDER_REF = {}


def _check_handle(env, cfg, n):
    """the handle runs the tracking kernel of the rule, and the render path of a small handle on the same config"""
    ri = env.render_info()
    per_thread, lanes = tracking_kernel(n, _sms())
    assert (ri["track_per_thread"], ri["track_lanes_per_env"]) == (per_thread, lanes), (n, ri)
    key = json.dumps(cfg, sort_keys=True)
    if key not in _RENDER_REF:
        small = _vec(cfg, 64)
        _RENDER_REF[key] = {k: small.render_info()[k] for k in _RENDER_KEYS}
        small.close()
    assert {k: ri[k] for k in _RENDER_KEYS} == _RENDER_REF[key], ("the render path depends on N", n, ri)
    return ri


# ------------------------------------------------------------------------------------------------ the nearest-laneline grid
class NearGrid:
    """numpy mirror of tc_build_near(map, 1.0, 16384) and tc_near_cell, and of the pre-filter's scan_limit (tc_pack.h): places
    cars in each regime of the laneline search and counts them. Only the counts depend on it; the oracle decides pass / fail."""

    def __init__(self, m):
        nodes = m.ll_nodes
        lo, hi = nodes.min(0), nodes.max(0)
        pad, max_cells = 1.0, 16384
        w, h = hi[0] - lo[0] + 2 * pad, hi[1] - lo[1] + 2 * pad
        self.cell = max(0.02, np.sqrt(w * h / max_cells))
        self.nx, self.ny = int(np.ceil(w / self.cell)), int(np.ceil(h / self.cell))
        self.x0, self.y0 = lo[0] - pad, lo[1] - pad
        self.inv = 1.0 / self.cell
        self.lo, self.hi = lo, hi
        self.scan_limit = 4.0 * max(1.0, np.abs(nodes).max(), np.abs(m.lp_nodes).max())

    def on_line(self, k, axis):
        """a coordinate whose cell coordinate is exactly the integer k (a cell line; 0 and nx / ny are the outer lines)"""
        o = self.x0 if axis == 0 else self.y0
        v = o + k * self.cell
        for _ in range(16):
            f = (v - o) * self.inv
            if f == k:
                return v
            v = np.nextafter(v, np.inf if f < k else -np.inf)
        return None

    def regimes(self, x, y):
        with np.errstate(invalid="ignore", over="ignore"):
            fx, fy = np.floor((x - self.x0) * self.inv), np.floor((y - self.y0) * self.inv)
            gx, gy = (x - self.x0) * self.inv, (y - self.y0) * self.inv
            inside = (fx >= 0) & (fx < self.nx) & (fy >= 0) & (fy < self.ny)
            far = ~((np.abs(x) <= self.scan_limit) & (np.abs(y) <= self.scan_limit))
            line = (gx == np.floor(gx)) | (gy == np.floor(gy))
            outer = (gx == 0) | (gx == self.nx) | (gy == 0) | (gy == self.ny)
        return {"grid": inside & ~line, "cell_line": inside & line & ~outer, "outer_line": outer & ~far,
                "near": ~inside & ~far & ~outer, "far": far}


def place_regime(grid, kind, rng):
    """(x, y) of one car in a regime of the laneline search"""
    g = grid
    if kind == "grid":
        return rng.uniform(g.lo[0], g.hi[0]), rng.uniform(g.lo[1], g.hi[1])
    if kind == "cell_line":
        for _ in range(64):
            x, y = g.on_line(int(rng.integers(1, g.nx)), 0), g.on_line(int(rng.integers(1, g.ny)), 1)
            if x is not None and y is not None:
                return x, y
        return g.x0 + 3.5 * g.cell, g.y0 + 3.5 * g.cell
    if kind == "outer_line":   # the grid's first column / row is inside, its far edge outside
        k = int(rng.integers(4))
        x = [g.on_line(0, 0), g.on_line(g.nx, 0)][k % 2] if k < 2 else rng.uniform(g.lo[0], g.hi[0])
        y = [g.on_line(0, 1), g.on_line(g.ny, 1)][k % 2] if k >= 2 else rng.uniform(g.lo[1], g.hi[1])
        return (g.x0 if x is None else x), (g.y0 if y is None else y)
    if kind == "near":        # about 1 m plus a fraction of a cell beyond the laneline bounding box
        s = rng.uniform(0.05, 0.95) * g.cell
        return [(g.x0 - s, rng.uniform(g.lo[1], g.hi[1])), (g.x0 + g.nx * g.cell + s, rng.uniform(g.lo[1], g.hi[1])),
                (rng.uniform(g.lo[0], g.hi[0]), g.y0 - s), (rng.uniform(g.lo[0], g.hi[0]), g.y0 + g.ny * g.cell + s)][int(rng.integers(4))]
    if kind == "far":         # beyond scan_limit: plain float64 scan; at 1e17 m every edge is at the same rounded distance (ties)
        return [(g.scan_limit + 5.0, rng.uniform(-3, 9)), (-rng.uniform(1, 3) * g.scan_limit, -g.scan_limit - 1.0),
                (3.0e17, -2.0e17)][int(rng.integers(3))]
    raise ValueError(kind)


REGIMES = ("grid", "cell_line", "outer_line", "near", "far")


# ------------------------------------------------------------------------------------------------ the scenario
def make_scenario(n, seed, grid, wheelbase):
    """T steps of events for n envs, independent of the state (so that one scenario drives several handles):
    cc / man actions; u-turn bursts (maneuver 2 for about half of the envs, every warp, after steps without 2); NaN actions in a
    few lanes of warp 0, in the last env and in the last full warp; cars placed in every regime of the laneline search while
    the env is wrapped (no termination), on lane 0 and 31 of warp 0 and on the last env among others, held still there;
    masked resets that select and deselect the last env; mark_done; reset_done."""
    rng = np.random.default_rng(seed)
    last = n - 1
    lw = (last // 32) * 32
    ev = []
    nan_envs = np.unique(np.array([3, 17, 29, last, max(lw - 32, 0) + 5, max(lw - 32, 0) + 31]) % n)
    placed = []
    for t in range(T):
        e = {"wrapped": 10 <= t < 15, "reset_mask": None, "reset_spawn": None, "place": None, "mark": None, "reset_done": t == 21}
        cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
        rev = rng.random(n) < 0.1
        cc[rev, 0] = -cc[rev, 0]
        man = rng.choice(np.array([0, 0, 1, 3], np.int32), n)
        if t in (2, 3, 8, 13, 17, 22):
            man[rng.random(n) < 0.5] = 2
            man[:32:3] = 2    # warp 0: eleven requests in one step
            man[lw:] = 2      # the last (partial) warp
        if t == 6:
            cc[nan_envs[::2], 0] = np.nan
            cc[nan_envs[1::2], 1] = np.nan
            man[nan_envs[: len(nan_envs) // 2]] = 2
        if t == 9:   # resets the NaN envs, selects the last env
            m = rng.random(n) < 0.2
            m[nan_envs] = True
            e["reset_mask"] = m
        if t in (10, 12):
            idx = np.unique(np.concatenate([[0, 31, 7, 13, 19, 25, lw, last], rng.choice(n, 48, replace=False)]) % n)
            shift = 0 if t == 10 else 2
            kinds = [REGIMES[(k + shift) % len(REGIMES)] for k in range(len(idx))]
            # lane 0, lane 31 and the last env leave the grid in both placements, each time in another regime
            for j, i in enumerate(idx):
                if i in (0, 31, last):
                    kinds[j] = ("near", "far")[(int(i == 31) + int(i == last) + shift // 2) % 2]
            xy = np.array([place_regime(grid, k, rng) for k in kinds], np.float64)
            rot = rng.uniform(-np.pi, np.pi, len(idx))
            rows = np.zeros((len(idx), 8))
            rows[:, 0], rows[:, 1], rows[:, 2] = xy[:, 0], xy[:, 1], rot
            rows[:, 5] = xy[:, 0] + wheelbase * np.cos(rot)
            rows[:, 6] = xy[:, 1] + wheelbase * np.sin(rot)
            e["place"] = (idx, rows)
            placed.append(idx)
        if 10 <= t < 15 and placed:   # the placed cars stand still (velocity 0, steering 0) while wrapped
            hold = np.unique(np.concatenate(placed))
            cc[hold] = 0
            man[hold] = 0
        if t == 18:
            m = rng.random(n) < 0.1
            m[last] = True
            e["mark"] = m
        if t == 20:   # deselects the last env
            m = rng.random(n) < 0.3
            m[0], m[last] = True, False
            e["reset_mask"] = m
        e["cc"], e["man"] = cc, man
        ev.append(e)
    return ev


def tile_scenario(ev, n, k):
    """the scenario of n envs for k*n envs: replica j + m*n of env j gets env j's events"""
    out = []
    for e in ev:
        f = dict(e)
        f["cc"], f["man"] = np.tile(e["cc"], (k, 1)), np.tile(e["man"], k)
        for key in ("reset_mask", "mark"):
            if e[key] is not None:
                f[key] = np.tile(e[key], k)
        if e["place"] is not None:
            idx, rows = e["place"]
            f["place"] = (np.concatenate([idx + m * n for m in range(k)]), np.tile(rows, (k, 1)))
        out.append(f)
    return out


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t if dtype is None else t.to(dtype)).cuda()


def place_cars(env, idx, rows):
    st = env.state_dict()
    sf = st["sf"]
    sf[_dev(idx).long()] = _dev(rows)
    env.load_state_dict({"sf": sf, "si": st["si"]})


# ------------------------------------------------------------------------------------------------ checks against the oracle
def oracle_frames(oenv, idx):
    """the oracle's frame of each env in idx at its current state"""
    out = np.zeros((len(idx),) + oenv.obs_shape, np.uint8)
    L = orc.lib()
    for k, i in enumerate(idx):
        L.orc_capture_frame(oenv.map.handle, orc._p(oenv.cam[i], orc._dp), oenv.H, oenv.W, int(oenv.thick[i]), orc._p(oenv.map.colors, orc._up),
                            orc._p(oenv.sf[i], orc._dp), oenv.fmt, orc._p(out[k], orc._up), None, None, None, None)
    return out


def check_frames(env, oenv, idx, where, stats, chunk=2048):
    idx = np.asarray(idx, np.int64)
    for s in range(0, len(idx), chunk):
        part = idx[s:s + chunk]
        got = env.obs[_dev(part)].cpu().numpy()
        want = oracle_frames(oenv, part)
        bad = np.nonzero((got != want).reshape(len(part), -1).any(axis=1))[0]
        assert len(bad) == 0, f"{where}: {len(bad)} of {len(part)} frames differ from the oracle, first env {int(part[bad[0]])}"
    stats["frames"] += len(idx)


def check_tracking(env, oenv, keep, where, lp_edges):
    """_compare_batch's checks (test_gpu_parity) on the envs in `keep`, plus the local path exports and the device-only
    edge ids; the frames are checked separately"""
    k = keep
    st = env.state_dict()
    sf, si = st["sf"].cpu().numpy(), st["si"].cpu().numpy()
    np.testing.assert_allclose(sf[k, :7], oenv.sf[k, :7], rtol=RTOL64, atol=1e-11, err_msg=f"state {where}")
    assert np.array_equal(si[k, :10], oenv.si[k, :10]), f"local path {where}"
    out = {key: v.cpu().numpy() for key, v in env.out.items()}
    np.testing.assert_allclose(out["info_f64"][k], oenv.info[k], rtol=RTOL64, atol=1e-11, err_msg=f"info {where}")
    assert np.array_equal(out["nearest_edge"][k], oenv.nearest[k]), f"nearest laneline edge {where}"
    assert np.array_equal(out["terminated"][k], oenv.terminated[k]), f"terminated {where}"
    assert np.array_equal(out["truncated"][k], oenv.truncated[k]), f"truncated {where}"
    np.testing.assert_allclose(out["cte"][k], oenv.cte[k], rtol=RTOL32, atol=1e-7)
    np.testing.assert_allclose(out["heading_error"][k], oenv.heading_error[k], rtol=RTOL32, atol=1e-7)
    np.testing.assert_allclose(out["laneline_distances"][k], oenv.dist[k], rtol=RTOL32, atol=1e-7)
    np.testing.assert_allclose(out["position"][k], oenv.sf[k, :2], rtol=RTOL32, atol=1e-7)
    # local_path_nodes / path_len against the oracle's si
    plen = oenv.si[k, 0]
    assert np.array_equal(out["path_len"][k], plen), f"path_len {where}"
    want = np.where((np.arange(8)[None, :] >> 1) < plen[:, None], oenv.si[k, 2:10], -1)
    assert np.array_equal(out["local_path_nodes"][k].reshape(-1, 8), want), f"local_path_nodes {where}"
    # the edge ids (device only) name the node pairs of the path
    for j in range(4):
        live = k & (si[:, 0] > j)
        e = si[live, 10 + j]
        assert ((e >= 0) & (e < len(lp_edges))).all(), f"edge id {j} out of range {where}"
        assert np.array_equal(lp_edges[e], si[live, 2 + 2 * j:4 + 2 * j]), f"edge id {j} does not name its node pair {where}"
    return sf, si


class CountingSampler:
    """SpawnSampler with the number of bounded draws each table entry took (a draw that lands on a node without successor is
    drawn again, map.py:61-64)"""

    def __init__(self, tables, n, K, seed):
        from tinycarlo_b200.spawn import SpawnSampler

        class _Counting:
            def __init__(self, rng):
                self.rng, self.calls = rng, np.zeros(n, np.int64)

            def bounded(self, k, m):
                self.calls[m] += 1
                return self.rng.bounded(k, m)

        tries = []

        class _S(SpawnSampler):
            def _draw(self, m):
                if not isinstance(self.rng, _Counting):
                    self.rng = _Counting(self.rng)
                before = self.rng.calls.copy()
                out = super()._draw(m)
                tries.append(self.rng.calls - before)
                return out
        self.table = _S(tables, n, table_len=K).seed(seed)
        self.tries = np.stack(tries, 1)   # [n, K]

    def redraws(self, used):
        """redraws among the first used[i] draws of every env"""
        cols = np.arange(self.tries.shape[1])[None, :] < used[:, None]
        return int(((self.tries - 1) * cols).sum())


# ------------------------------------------------------------------------------------------------ part 2: oracle parity
CASES = [("warp_partial", "default"), ("warp_last", None), ("group8_first", None), ("group8_last", "default"),
         ("thread_first", "default"), ("thread_big", None)]


@pytest.mark.parametrize("case,spawn", CASES, ids=[f"{c}-{'spawn_points' if s else 'any_node'}" for c, s in CASES])
def test_tracking_kernel_matches_oracle(case, spawn):
    """Knuffingen, 64x96 classes, next-step autoreset, the scenario of make_scenario: every step, every env against the oracle
    (NaN envs excepted until their reset; their outputs are compared across kernels in test_tracking_kernels_are_bit_identical)."""
    n = _count(case)
    cfg = make_config("knuffingen", "classes", cam={"resolution": RES}, spawn=spawn)
    env = _vec(cfg, n, autoreset="next_step")
    ri = _check_handle(env, cfg, n)
    oenv = oracle_env(cfg, n)
    m = env.map
    lp_edges = np.asarray(m.lp_edges)
    grid = NearGrid(m)
    seed = zlib.crc32(f"{case}{spawn}".encode()) & 0xFFFF
    ev = make_scenario(n, seed, grid, float(env._car_rows[0, 0]))
    draws = CountingSampler(m, n, SPAWN_TABLE, seed)
    n_drawn = np.ones(n, np.int64)
    stats = {"frames": 0}
    cnt = {"uturn_scans": 0, "uturn_max_per_warp": 0, "uturn_warps_2plus": 0, "uturn_no_edge": 0, "autoresets": 0, "resets": 0,
           **{f"cars_{r}": 0 for r in REGIMES}, "offgrid_lane0": 0, "offgrid_lane31": 0, "offgrid_last": 0}
    block = FOUR_BLOCK[ri["track_lanes_per_env"]]
    cnt["partial_block_envs"] = n % block
    all_envs = np.arange(n)
    tail = all_envs[-256:]
    tainted = np.zeros(n, bool)   # NaN actions: the oracle clips NaN to -1 where np.clip (and the device) propagate it

    def check_draws(where):
        assert (n_drawn <= SPAWN_TABLE).all()
        assert np.array_equal(env._spawn_nodes.cpu().numpy(), draws.table[all_envs, n_drawn - 1]), f"device spawn draw {where}"

    env.reset(seed=seed)
    check_draws("reset")
    oenv.reset(draws.table[:, 0], render=False)
    check_frames(env, oenv, all_envs, "reset", stats)
    for t, e in enumerate(ev):
        if e["wrapped"] != env.wrapped:
            env.set_wrapped(e["wrapped"])
            oenv.wrapped = e["wrapped"]
        if e["reset_mask"] is not None:
            mk = e["reset_mask"]
            env.reset(mask=torch.from_numpy(mk))
            n_drawn[mk] += 1
            check_draws(f"masked reset before step {t}")
            oenv.reset(draws.table[all_envs, n_drawn - 1], mask=mk.astype(np.uint8), render=False)
            tainted[mk] = False
            cnt["resets"] += int(mk.sum())
            st = env.state_dict()
            np.testing.assert_allclose(st["sf"].cpu().numpy()[:, :7], oenv.sf[:, :7], rtol=RTOL64, atol=1e-11)
            check_frames(env, oenv, np.nonzero(mk)[0], f"masked reset before step {t}", stats)
        if e["place"] is not None:
            idx, rows = e["place"]
            place_cars(env, idx, rows)
            oenv.sf[idx] = rows
        if e["mark"] is not None:
            env.mark_done(torch.from_numpy(e["mark"]))
        done = env.done_flags.cpu().numpy().astype(bool)
        si0 = env.state_dict()["si"].cpu().numpy()
        # u-turn scans this step starts (tc_wants_uturn_scan on the state before the step)
        valid = (si0[:, 0] > 0) & (si0[:, 10] >= 0) & (si0[:, 10] < len(lp_edges)) & (si0[:, 2] >= 0) & (si0[:, 3] >= 0)
        want = (e["man"] == 2) & (si0[:, 1] != 2) & valid & ~done
        per_warp = np.bincount(all_envs[want] // 32, minlength=(n + 31) // 32)
        cnt["uturn_scans"] += int(want.sum())
        cnt["uturn_max_per_warp"] = max(cnt["uturn_max_per_warp"], int(per_warp.max()))
        cnt["uturn_warps_2plus"] += int((per_warp >= 2).sum())
        env.step({"car_control": _dev(e["cc"]), "maneuver": _dev(e["man"])})
        n_drawn[done] += 1
        keep_sf, keep_si = oenv.sf.copy(), oenv.si.copy()
        oenv.step(e["cc"].astype(np.float64), e["man"], render=False)
        if done.any():   # next-step autoreset on the oracle: the finished envs are reset on the nodes the device drew
            oenv.sf[done], oenv.si[done] = keep_sf[done], keep_si[done]
            oenv.reset(draws.table[all_envs, n_drawn - 1], mask=done.astype(np.uint8), render=False)
            oenv.info[done] = 0
            oenv.nearest[done] = -1
            oenv.terminated[done] = 0
            oenv.truncated[done] = 0
            cnt["autoresets"] += int(done.sum())
            tainted[done] = False
        assert np.array_equal(env.reset_mask.cpu().numpy(), done), f"reset mask step {t}"
        tainted |=~np.isfinite(e["cc"]).all(1)
        keep = ~tainted
        sf, si = check_tracking(env, oenv, keep, f"step {t}", lp_edges)
        check_draws(f"step {t}")
        cnt["uturn_no_edge"] += int((want & keep & (oenv.truncated == 1) & (oenv.si[:, 1] == si0[:, 1])).sum())
        dev_done = env.done_flags.cpu().numpy().astype(bool)
        assert np.array_equal(dev_done[keep], (oenv.terminated | oenv.truncated)[keep].astype(bool)), f"done flags step {t}"
        # laneline-search regimes of the cars that searched this step
        searched = keep & (si[:, 0] >= 2) & ~done
        reg = grid.regimes(sf[:, 0], sf[:, 1])
        for r in REGIMES:
            cnt[f"cars_{r}"] += int((reg[r] & searched).sum())
        off = (reg["near"] | reg["far"]) & searched
        cnt["offgrid_lane0"] += int(off[0])
        cnt["offgrid_lane31"] += int(off[31 % n])
        cnt["offgrid_last"] += int(off[n - 1])
        # frames: every env every 5th step, the envs this step reset and the last 256 envs every step
        frames = all_envs[keep] if t % 5 == 0 else np.union1d(tail[keep[tail]], np.nonzero(done & keep)[0])
        check_frames(env, oenv, frames, f"step {t}", stats)
        if e["reset_done"]:
            fin = (env.out["terminated"] | env.out["truncated"]).cpu().numpy().astype(bool)
            env.reset_done()
            n_drawn[fin] += 1
            check_draws(f"reset_done after step {t}")
            oenv.reset(draws.table[all_envs, n_drawn - 1], mask=fin.astype(np.uint8), render=False)
            tainted[fin] = False
            cnt["resets"] += int(fin.sum())
            check_frames(env, oenv, np.nonzero(fin)[0], f"reset_done after step {t}", stats)
    cnt["spawn_redraws"] = draws.redraws(n_drawn)
    print(f"{case} ({'spawn_points' if spawn else 'any node'}): {_kernel_name(ri)}, {n} envs, {stats['frames']} frames, {cnt}")
    # coverage floors: a later edit of the scenario must not quietly stop reaching these paths
    assert cnt["uturn_scans"] >= n and cnt["uturn_max_per_warp"] >= 8 and cnt["uturn_warps_2plus"] >= (n // 32) * 3, cnt
    assert cnt["autoresets"] >= n // 20 and cnt["resets"] >= n // 4, cnt
    if spawn is None:
        assert cnt["spawn_redraws"] >= 1, cnt
    for r in REGIMES:
        assert cnt[f"cars_{r}"] >= 3, (r, cnt)
    assert cnt["offgrid_lane0"] >= 2 and cnt["offgrid_lane31"] >= 2 and cnt["offgrid_last"] >= 2, cnt
    if case != "warp_last":
        assert cnt["partial_block_envs"] > 0, cnt
    env.close()


# ------------------------------------------------------------------------------------------------ u-turn without an edge
def _triangle_map(path):
    """Knuffingen's lanelines with a one-way triangular lanepath: its edges point at 0, 120 and 240 degrees, so a u-turn
    (the reverse direction +-30 degrees) finds no edge from anywhere. No bundled map has such an edge: Knuffingen's lanepath
    has one within +-30 degrees of the reverse of every edge."""
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tinycarlo_b200", "maps", "knuffingen.json")) as f:
        data = json.load(f)
    ppm = PPM["knuffingen"]
    tri = [(2.0, 1.0), (6.0, 1.0), (4.0, 1.0 + 2.0 * np.sqrt(3.0))]
    data["lanepath"] = {"layer_color": data["lanepath"].get("layer_color", [0, 0, 0]), "nodes": [[x * ppm, y * ppm] for x, y in tri],
                        "edges": [[0, 1], [1, 2], [2, 0]]}
    with open(path, "w") as f:
        json.dump(data, f)
    return path


@pytest.mark.parametrize("case", ["warp_partial", "group8_first", "thread_first"])
def test_uturn_without_edge_truncates(case, tmp_path):
    """maneuver 2 after another maneuver with no lanepath edge within +-30 degrees of the reverse direction: truncated, the
    local path and the last maneuver untouched (DESIGN.md section 2), requested by about half of every warp's envs at once"""
    n = _count(case)
    path = _triangle_map(str(tmp_path / "triangle.json"))
    cfg = make_config("knuffingen", "classes", cam={"resolution": RES})
    cfg["map"] = {"json_path": path, "pixel_per_meter": PPM["knuffingen"], "spawn_points": [0, 1, 2]}
    env = _vec(cfg, n)
    ri = _check_handle(env, cfg, n)
    cc_ = cfg["camera"]
    E, K = orc.camera_matrices(cc_["position"], cc_["orientation"], cc_["fov"], RES)
    oenv = orc.OracleVecEnv(orc.OracleMap(path, PPM["knuffingen"], [0, 1, 2]), n, orc.pack_car(cfg["car"], cfg["sim"]["fps"]),
                            orc.pack_cam(E, K, cc_["max_range"]), cc_["line_thickness"], RES[0], RES[1], "classes")
    lp_edges = np.asarray(env.map.lp_edges)
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    env.reset(seed=7)
    oenv.reset(env._spawn_nodes.cpu().numpy(), render=False)
    stats = {"frames": 0}
    check_frames(env, oenv, np.arange(n), "reset", stats)
    failed, max_warp = 0, 0
    for t in range(6):
        cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-0.3, 0.3, n)], 1).astype(np.float32)
        man = np.where(rng.random(n) < 0.5, 2, 0).astype(np.int32)
        man[-1] = 2
        si0 = env.state_dict()["si"].cpu().numpy()
        want = (man == 2) & (si0[:, 1] != 2) & (si0[:, 0] > 0)
        env.step({"car_control": _dev(cc), "maneuver": _dev(man)})
        oenv.step(cc.astype(np.float64), man, render=False)
        sf, si = check_tracking(env, oenv, np.ones(n, bool), f"step {t}", lp_edges)
        trunc = env.out["truncated"].cpu().numpy().astype(bool)
        assert trunc[want].all(), f"a u-turn without an edge must truncate (step {t})"
        assert np.array_equal(si[want], si0[want]), f"a u-turn without an edge must leave the path untouched (step {t})"
        failed += int(want.sum())
        max_warp = max(max_warp, int(np.bincount(np.nonzero(want)[0] // 32).max()))
        check_frames(env, oenv, np.arange(n)[-256:], f"step {t}", stats)
    print(f"{case}: {_kernel_name(ri)}, {n} envs, {failed} u-turns without an edge, at most {max_warp} in one warp in one step")
    assert failed >= n and max_warp >= 8
    env.close()


# ------------------------------------------------------------------------------------------------ part 3: bit-identical kernels
def _bits(t):
    """a tensor as its bit patterns (NaNs compare by payload, -0.0 differs from 0.0)"""
    return t.view({8: torch.int64, 4: torch.int32, 2: torch.int16}[t.element_size()]) if t.is_floating_point() else t


def _replicas_equal(base, big, k, what):
    b = _bits(base)
    g = _bits(big).reshape((k,) + tuple(b.shape))
    same = (g == b.unsqueeze(0)).reshape(k, b.shape[0], -1).all(-1)
    if not bool(same.all()):
        r, j = (~same).nonzero()[0].tolist()
        raise AssertionError(f"{what}: replica {r} of env {j} differs from the base handle")


def _snapshot(env):
    st = env.state_dict()
    s = {"sf": st["sf"], "si": st["si"], "obs": env.obs, "spawn_nodes": env._spawn_nodes, "spawn_rng": env._rng_state,
         "done": env.done_flags, "reset_mask": env._reset_mask}
    s.update({f"out.{k}": v for k, v in env.out.items()})
    return s


def test_tracking_kernels_are_bit_identical():
    """DESIGN.md section 4: the thread-per-env kernel's results are bit-identical to the lane-group kernels'. B envs on the
    warp-per-env kernel, 2B on 8 lanes per env and 9B on the thread kernel (1771, 3542, 15939 on a B200, all with partial last
    blocks), replica j + m*B of env j restored from the same checkpoint (state, spawn streams) and driven by the same events:
    every replica equals its env of the B handle exactly, NaN envs included, after every reset and every step."""
    sms = _sms()
    B = kernel_counts(sms)["warp_partial"]
    ks = [1, 2, 9]
    assert [tracking_kernel(k * B, sms) for k in ks] == [(0, 32), (0, 8), (1, 1)], B
    cfg = make_config("knuffingen", "classes", cam={"resolution": RES}, spawn=None)
    envs = [_vec(cfg, k * B, autoreset="next_step") for k in ks]
    kernels = [_kernel_name(_check_handle(e, cfg, k * B)) for e, k in zip(envs, ks)]
    grid = NearGrid(envs[0].map)
    ev = make_scenario(B, 4242, grid, float(envs[0]._car_rows[0, 0]))
    base = envs[0]
    base.reset(seed=11)
    for _ in range(3):   # a few steps so that the checkpoint is not a spawn state
        base.step({"car_control": _dev(ev[0]["cc"]), "maneuver": _dev(np.zeros(B, np.int32))})
    ck = base.checkpoint()
    for e, k in zip(envs[1:], ks[1:]):
        e.reset(seed=99)
        e.restore({key: (v.repeat(k, *([1] * (v.dim() - 1)))) for key, v in ck.items()})
    compared = 0

    def compare(where, keys=None):
        nonlocal compared
        torch.cuda.synchronize()
        s0 = _snapshot(base)
        for e, k in zip(envs[1:], ks[1:]):
            s = _snapshot(e)
            for key in keys or s0:
                _replicas_equal(s0[key], s[key], k, f"{key} ({_kernel_name(e.render_info())}, {where})")
            compared += 1

    # the base handle's outputs are those of its last step, the replicas' those of their reset: compare what restore sets
    compare("restore", ("sf", "si", "obs", "spawn_nodes", "spawn_rng", "done"))
    nan_seen = False
    for t, e0 in enumerate(ev):
        for env, k in zip(envs, ks):
            e = tile_scenario([e0], B, k)[0]
            if e["wrapped"] != env.wrapped:
                env.set_wrapped(e["wrapped"])
            if e["reset_mask"] is not None:
                env.reset(mask=torch.from_numpy(e["reset_mask"]))
            if e["place"] is not None:
                place_cars(env, *e["place"])
            if e["mark"] is not None:
                env.mark_done(torch.from_numpy(e["mark"]))
            env.step({"car_control": _dev(e["cc"]), "maneuver": _dev(e["man"])})
        compare(f"step {t}")
        nan_seen |= bool(torch.isnan(base.state_dict()["sf"][:, 0]).any())
        if e0["reset_done"]:
            for env in envs:
                env.reset_done()
            compare(f"reset_done after step {t}")
    print(f"B = {B}: {kernels}, {compared} comparisons of every replica")
    assert nan_seen
    for e in envs:
        e.close()


# ------------------------------------------------------------------------------------------------ part 4: a rig on <8> and thread
@pytest.mark.parametrize("case", ["group8_first", "thread_first"])
def test_rig_on_the_larger_batch_kernels(case):
    """M = 2 (the config camera and a rear camera): both tracking kernels write the poses of every view and, on a masked reset,
    the mask of every view. The buffer is poisoned with 0xAB before the reset; the views of deselected envs (the last env among
    them) keep the poison, a selected env whose reset fails (dead-end spawn node) is rendered at its old pose, and every other
    view equals the oracle's frame for its camera row."""
    n = _count(case)
    M = 2
    cfg = make_config("knuffingen", "classes", cam={"resolution": RES})
    plain = dict(cfg)
    cfg = dict(cfg, cameras=[{}, REAR])
    env = _vec(cfg, n)
    ri = _check_handle(env, cfg, n)
    assert env.obs.shape[:2] == (n, M)
    oenv = oracle_env(plain, n)
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    H, W = RES

    L = orc.lib()

    def check_views(envs, where):
        got = env.obs[_dev(envs)].flatten(0, 1).cpu().numpy()
        views = [int(i) * M + m for i in envs for m in range(M)]
        want = np.zeros((len(views), oenv.map.C, H, W), np.uint8)
        for k, v in enumerate(views):   # rig_util.oracle_views, for the compared views only
            L.orc_capture_frame(oenv.map.handle, orc._p(env._cam_rows[v], orc._dp), H, W, int(env._thickness[v]), orc._p(oenv.map.colors, orc._up),
                                orc._p(oenv.sf[v // M], orc._dp), 0, orc._p(want[k], orc._up), None, None, None, None)
        bad = np.nonzero((got != want).reshape(len(views), -1).any(axis=1))[0]
        assert len(bad) == 0, f"{where}: {len(bad)} of {len(views)} views differ; first view {views[bad[0]]}"
        return len(views)

    env.reset(seed=5)
    oenv.reset(env._spawn_nodes.cpu().numpy(), render=False)
    frames = 0
    for t in range(4):
        if t == 2:
            for r in range(2):   # two masked resets with different masks: a stale view mask would show in the second
                mask = rng.random(n) < (0.4 if r == 0 else 0.25)
                mask[0], mask[n - 1] = True, False
                nodes = env._spawn_nodes.cpu().numpy().copy()
                sel = np.nonzero(mask)[0]
                nodes[sel] = rng.choice(np.array([18, 156, 217, 214], np.int32), len(sel))
                failed = sel[:: 7]
                nodes[failed] = DEAD_END
                env.obs.view(torch.uint8).fill_(0xAB)
                env.reset(mask=torch.from_numpy(mask), spawn_nodes=torch.from_numpy(nodes))
                oenv.reset(nodes, mask=mask.astype(np.uint8), render=False)
                raw = env.obs.view(torch.uint8).reshape(n, -1)
                assert bool((raw[_dev(np.nonzero(~mask)[0])] == 0xAB).all()), f"a masked reset wrote views of deselected envs ({r})"
                np.testing.assert_allclose(env.state_dict()["sf"].cpu().numpy()[:, :7], oenv.sf[:, :7], rtol=RTOL64, atol=1e-11)
                frames += check_views(sel, f"masked reset {r}")
                assert len(failed) > 0
        cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
        man = rng.integers(0, 4, n).astype(np.int32)
        env.obs.view(torch.uint8).fill_(0xAB)
        env.step({"car_control": _dev(cc), "maneuver": _dev(man)})
        oenv.step(cc.astype(np.float64), man, render=False)
        np.testing.assert_allclose(env.state_dict()["sf"].cpu().numpy()[:, :7], oenv.sf[:, :7], rtol=RTOL64, atol=1e-11)
        views = np.arange(n) if t == 3 else np.unique(np.concatenate([np.arange(64), np.arange(n)[-256:]]))
        frames += check_views(views, f"step {t}")
    print(f"{case}: {_kernel_name(ri)}, {n} envs x {M} views, {frames} views compared")
    env.close()
