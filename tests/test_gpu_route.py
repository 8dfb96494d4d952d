"""The navigation goals on the device (config section `navigation`, tc_route_kernel) against the numpy restatement of the
contract (tests/route_util.py) fed with the device state, every env and every step; an autopilot that follows route_command to
its goal; and what switching the feature on must leave alone: observations, info, BEV, range scan, reward and flags, spawn
nodes, one launch more per step and reset, guard bands, env counts, every entry point that launches the kernel, graph
replay, checkpoint / restore, set_goals, a camera rig, the grouped and the single env."""
import numpy as np
import pytest
import torch

import route_util as R
from rig_util import REAR
from tinycarlo_b200 import TinyCarloEnv, TinyCarloVecEnv
from tinycarlo_b200.config import make_config
from tinycarlo_b200.grouped_env import TinyCarloGroupedVecEnv
from tinycarlo_b200.spawn import stream_seeds
from tinycarlo_b200.wrapper import RouteProgressRewardWrapper

pytestmark = pytest.mark.gpu

KEYS = ("goal", "goal_position", "route_command", "route_distance", "route_progress", "goal_reached")


def nav_config(map_name, nav=None, car=None, extra=None):
    cfg = make_config(map_name, "classes", car=car)
    if nav is not None:
        cfg["navigation"] = dict(nav)
    cfg.update(extra or {})
    return cfg


def stanley(info, max_steer, speed=0.8, k=4.0):
    """examples/stanley_control.py:56-58 as bench.py states it, with maneuver = route_command (-1: straight)"""
    n = info["cte"].shape[0]
    cc = torch.empty((n, 2), dtype=torch.float32, device=info["cte"].device)
    cc[:, 0] = speed
    cc[:, 1] = (info["heading_error"] + torch.atan2(k * info["cte"], torch.full_like(info["cte"], speed))) * (180 / np.pi / max_steer)
    man = info["route_command"].clamp(min=0) if "route_command" in info else torch.zeros(n, dtype=torch.int32, device=cc.device)
    return {"car_control": cc, "maneuver": man.to(torch.int32)}


def random_actions(rng, n, dev):
    cc = np.stack([rng.uniform(0.2, 1.0, n), rng.uniform(-1.0, 1.0, n)], 1).astype(np.float32)
    return {"car_control": torch.from_numpy(cc).to(dev), "maneuver": torch.from_numpy(rng.choice([0, 1, 2, 3], n).astype(np.int32)).to(dev)}


class Oracle:
    """route_util.update() fed with the env's device state after every call"""

    def __init__(self, env, seed):
        self.env = env
        nv = env.nav_cfg
        self.goals, self.reach, self.on_reach = list(nv["goals"]), nv["reach_radius"], 1 if nv["on_reach"] == "terminate" else 0
        self.D, self.cmd = R.route_table(env.map, self.goals)
        self.gens = R.generators(stream_seeds(env.num_envs, seed, env.env_index_offset))
        n = env.num_envs
        self.k, self.prev = np.full(n, -1, np.int64), np.full(n, np.inf)

    def check(self, mode, mask=None, was_reset=None):
        e = self.env
        st = e.state_dict()
        sf, si = st["sf"].cpu().numpy(), st["si"].cpu().numpy()
        want = R.update(e.map, self.D, self.cmd, self.goals, self.reach, self.on_reach, mode, sf, si, self.gens, self.k, self.prev,
                        mask=mask, was_reset=was_reset)
        got = {k: v.cpu().numpy() for k, v in e.route.items()}
        R.assert_outputs_equal(got, want, what=f"mode {mode}")
        assert np.array_equal(e._goal_index.cpu().numpy(), self.k)
        assert np.array_equal(e._prev_distance.cpu().numpy().view(np.int64), self.prev.view(np.int64))
        assert np.array_equal(e._goal_rng.cpu().numpy().view(np.uint64), R.generator_rows(self.gens))
        return want


@pytest.mark.parametrize("on_reach", ["resample", "terminate"])
@pytest.mark.parametrize("map_name", ["knuffingen", "simple_layout"])
def test_route_rollout_matches_oracle(map_name, on_reach):
    """reset, 120 Stanley steps following the route with next-step autoresets (a quarter marked done at step 5), a masked reset"""
    n, seed = 512, 4
    env = TinyCarloVecEnv(nav_config(map_name, {"on_reach": on_reach, "reach_radius": 0.08}, car={"max_velocity": 1.0}), n,
                          device="cuda:0", autoreset="next_step")
    env.no_observation = True
    env.reset(seed=seed)
    orc = Oracle(env, seed)
    orc.check(1)
    info = env._info()
    reaches = autoresets = draws = 0
    for t in range(120):
        if t == 5:
            env.mark_done(torch.from_numpy(np.arange(n) % 4 == 0).to(env.device))
        _, _, term, trunc, info = env.step(stanley(info, 30))
        was = env.reset_mask.cpu().numpy()
        want = orc.check(0, was_reset=was)
        tflag = np.array([bool(v) for v in want["terminate"]])
        if on_reach == "terminate":
            assert term.cpu().numpy()[tflag].all() and env.done_flags.cpu().numpy().astype(bool)[tflag].all()
        reaches += int(np.sum([bool(v) for v in want["reached"]]))
        autoresets += int(was.sum())
        draws += int(was.sum())
    mask = np.random.default_rng(1).random(n) < 0.5
    env.reset(mask=torch.from_numpy(mask))
    orc.check(1, mask=mask)
    print(f"{map_name} {on_reach}: {reaches} goals reached, {autoresets} autoresets")
    assert reaches > 0 and autoresets >= n // 4


def test_route_autopilot_reaches_goals():
    """Stanley with maneuver = route_command: 90 % of the envs that neither terminated nor truncated reach their goal within
    2 * initial distance / (speed * max_velocity * dt) + 60 steps"""
    n = 1024
    mv, speed, fps = 0.3, 0.8, 30
    env = TinyCarloVecEnv(nav_config("knuffingen", {"on_reach": "terminate", "reach_radius": 0.1}, car={"max_velocity": mv}), n,
                          device="cuda:0")
    env.no_observation = True
    _, info = env.reset(seed=12)
    d0 = env.route["distance"].cpu().numpy().astype(np.float64)
    has_goal = env.route["goal"].cpu().numpy() >= 0
    bound = np.where(np.isfinite(d0), 2 * d0 / (speed * mv / fps) + 60, 0).astype(np.int64)
    reached_at = np.full(n, -1)
    failed = np.zeros(n, bool)
    for t in range(int(bound[has_goal].max()) + 1):
        _, _, term, trunc, info = env.step(stanley(info, 30, speed))
        r = info["goal_reached"].cpu().numpy()
        bad = (term.cpu().numpy() | trunc.cpu().numpy()) & ~r
        reached_at[(reached_at < 0) & r & ~failed] = t
        failed |= bad & (reached_at < 0)
    ok = has_goal & ~failed
    in_time = (reached_at >= 0) & (reached_at <= bound)
    frac, frac_any = float(in_time[ok].mean()), float((reached_at[ok] >= 0).mean())
    print(f"autopilot: {ok.sum()} of {n} envs drove undisturbed, {frac:.4f} of them reached their goal within the bound, "
          f"{frac_any:.4f} within the run ({(has_goal & failed).sum()} left the road or lost their path)")
    assert ok.sum() > n // 4
    late = ok & ~in_time
    print(f"autopilot: {late.sum()} undisturbed envs missed their bound; final route_distance of those "
          f"{np.round(info['route_distance'].cpu().numpy()[late][:10], 3)}")
    assert frac >= 0.9   # the rest overshoot the goal node outside the radius at a junction and are routed round again


def test_route_changes_nothing_else():
    """obs, info, BEV, range scan, reward and flags equal a run without the section; spawn nodes equal; one launch more per
    step and per reset; terminate mode only ORs the reach into the flags"""
    n = 300
    extra = {"bev": {}, "lidar": {"rays": 16}}
    envs = [TinyCarloVecEnv(nav_config("knuffingen", nav, extra=extra), n, device="cuda:0", autoreset="next_step")
            for nav in (None, {}, {"on_reach": "terminate", "reach_radius": 0.2})]
    rng = np.random.default_rng(3)
    outs = []
    for e in envs:
        l0 = e.launch_count
        e.reset(seed=9)
        outs.append([e.launch_count - l0])
    assert outs[1][0] == outs[0][0] + 1 and outs[2][0] == outs[0][0] + 1
    acts = [random_actions(rng, n, envs[0].device) for _ in range(40)]
    diverged = False   # terminate mode changes which envs autoreset: its states part ways after the first reach
    for t, a in enumerate(acts):
        res = []
        for e in envs:
            l0 = e.launch_count
            obs, rew, term, trunc, info = e.step(a)
            res.append((e.launch_count - l0, obs.clone(), rew.clone(), term.clone(), trunc.clone(), {k: v.clone() for k, v in info.items()},
                        e._spawn_nodes.clone(), e.reset_mask.clone()))
        base = res[0]
        for j, r in enumerate(res[1:], 1):
            assert r[0] == base[0] + 1
            assert set(r[5]) == set(base[5]) | set(KEYS)
            if j == 2 and diverged:
                continue
            assert torch.equal(r[1], base[1]) and torch.equal(r[2], base[2]) and torch.equal(r[4], base[4])
            assert torch.equal(r[6], base[6]) and torch.equal(r[7], base[7])
            for k, v in base[5].items():
                assert torch.equal(r[5][k], v), k
            if j == 1:
                assert torch.equal(r[3], base[3])
            else:
                assert torch.equal(r[3], base[3] | r[5]["goal_reached"])
                diverged = bool(r[5]["goal_reached"].any())
    assert not set(KEYS) & set(base[5])


@pytest.mark.parametrize("n", [1, 4099, 16384])
def test_route_env_counts_and_guard_bands(n):
    """outputs written for every env and nowhere else, equal to the oracle"""
    env = TinyCarloVecEnv(nav_config("knuffingen", {}), n, device="cuda:0", autoreset="next_step")
    env.no_observation = True
    G = 1 << 12
    guards = {}
    for k, v in list(env.route.items()):
        flat = v.reshape(-1)
        buf = torch.full((flat.numel() + 2 * G,), 0x5A, dtype=flat.dtype, device=env.device) if flat.dtype != torch.float32 else \
            torch.full((flat.numel() + 2 * G,), -123.0, dtype=flat.dtype, device=env.device)
        guards[k] = buf
        env.route[k] = buf[G:G + flat.numel()].view(v.shape)
    import ctypes as C
    from tinycarlo_b200 import _lib
    nv = env.nav_cfg
    rdesc = _lib.TcRouteDesc(len(env._nav_goals), env._nav_goals.ctypes.data, nv["reach_radius"], 0)
    routs = _lib.TcRouteOutputs(*(env.route[k].data_ptr() for k in _lib.ROUTE_OUTPUT_FIELDS))
    _lib.check(env._L.tc_set_route(env._h, C.byref(rdesc), C.c_void_p(env._goal_rng.data_ptr()), C.c_void_p(env._goal_index.data_ptr()),
                                   C.c_void_p(env._prev_distance.data_ptr()), C.byref(routs)), "tc_set_route")
    env._info_cache = env._info()
    env.reset(seed=2)
    orc = Oracle(env, 2)
    orc.check(1)
    rng = np.random.default_rng(0)
    for t in range(3):
        env.step(random_actions(rng, n, env.device))
        orc.check(0, was_reset=env.reset_mask.cpu().numpy())
    for k, buf in guards.items():
        head, tail = buf[:G], buf[-G:]
        fill = 0x5A if buf.dtype != torch.float32 else -123.0
        assert (head == fill).all() and (tail == fill).all(), k


def test_route_entry_points():
    """tc_step_f64, step_host, a graph replay against eager steps, checkpoint / restore bit for bit, set_goals"""
    n = 256
    cfg = nav_config("knuffingen", {})
    a, b = (TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step") for _ in range(2))
    for e in (a, b):
        e.no_observation = True
        e.reset(seed=5)
    orc = Oracle(a, 5)
    orc.check(1)
    # float64 actions
    rng = np.random.default_rng(2)
    act = random_actions(rng, n, a.device)
    a.step({"car_control": act["car_control"].double(), "maneuver": act["maneuver"]})
    orc.check(0, was_reset=a.reset_mask.cpu().numpy())
    # step_host
    cc, man = act["car_control"].cpu(), act["maneuver"].cpu()
    rew, term, trunc = torch.zeros(n), torch.zeros(n, dtype=torch.uint8), torch.zeros(n, dtype=torch.uint8)
    a.step_host(cc, man, rew, term, trunc)
    orc.check(0, was_reset=a.reset_mask.cpu().numpy())
    # checkpoint, 30 steps, restore, the same 30 steps: bit for bit
    ck = a.checkpoint()
    acts = [random_actions(rng, n, a.device) for _ in range(30)]
    first = []
    for x in acts:
        a.step(x)
        first.append({k: v.clone() for k, v in a.route.items()})
    a.restore(ck)
    for x, f in zip(acts, first):
        a.step(x)
        for k, v in a.route.items():
            assert torch.equal(v.view(torch.uint8) if v.dtype == torch.float32 else v, f[k].view(torch.uint8) if v.dtype == torch.float32 else f[k]), k
    # graph replay against eager steps
    a.restore(ck)
    b.restore(ck)
    graph = b.capture(lambda e: act, steps=4, warmup=1)
    a.restore(ck)
    b.restore(ck)
    for _ in range(3):
        graph.replay()
        for _ in range(4):
            a.step(act)
    torch.cuda.synchronize()
    for k in a.route:
        assert torch.equal(a.route[k].nan_to_num(), b.route[k].nan_to_num()), k
    # set_goals: the goal list only
    goals = a.nav_cfg["goals"]
    nodes = torch.tensor([goals[i % len(goals)] for i in range(n)], dtype=torch.int32)
    mask = torch.from_numpy(np.arange(n) % 3 == 0)
    a.set_goals(nodes, mask)
    got = a.route["goal"].cpu().numpy()
    assert (got[mask.numpy()] == nodes.numpy()[mask.numpy()]).all()
    assert (a.route["progress"].cpu().numpy()[mask.numpy()] == 0).all()
    with pytest.raises(ValueError):
        a.set_goals(torch.full((n,), 0, dtype=torch.int32))


def test_route_rig_grouped_single_and_reward():
    cfg = nav_config("knuffingen", {})
    cfg["cameras"] = [{}, REAR]
    e = TinyCarloVecEnv(cfg, 64, device="cuda:0", autoreset="next_step")
    e.reset(seed=1)
    orc = Oracle(e, 1)
    orc.check(1)
    e.step(random_actions(np.random.default_rng(0), 64, e.device))
    orc.check(0, was_reset=e.reset_mask.cpu().numpy())
    # grouped: goals seeded by global env index, so the groups' goals equal those of one env of all 64
    cfg1 = nav_config("knuffingen", {})
    g = TinyCarloGroupedVecEnv(cfg1, [(40, [64, 64]), (24, [128, 160])], device="cuda:0")
    _, ginfo = g.reset(seed=7)
    full = TinyCarloVecEnv(cfg1, 64, device="cuda:0")
    _, finfo = full.reset(seed=7)
    for k in KEYS:
        assert torch.equal(ginfo[k].nan_to_num(), finfo[k].nan_to_num()), k
    # single env: Python scalars
    se = TinyCarloEnv(config=cfg1, device="cuda:0")
    _, info = se.reset(seed=3)
    obs, rew, term, trunc, info = se.step({"car_control": [0.5, 0.0], "maneuver": 0})
    assert isinstance(info["goal"], int) and isinstance(info["route_distance"], float) and isinstance(info["goal_reached"], bool)
    assert isinstance(info["goal_position"], list) and isinstance(info["route_command"], int)
    # the reward wrapper: progress_scale * route_progress + goal_bonus * goal_reached, 0 on autoreset steps
    w = RouteProgressRewardWrapper(TinyCarloVecEnv(cfg1, 64, device="cuda:0", autoreset="next_step"), progress_scale=10.0, goal_bonus=2.0)
    w.reset(seed=0)
    w.unwrapped.mark_done(torch.from_numpy(np.arange(64) % 2 == 0).to(w.unwrapped.device))
    _, r, *_ , info = w.step(random_actions(np.random.default_rng(1), 64, w.unwrapped.device))
    exp = 10.0 * info["route_progress"] + 2.0 * info["goal_reached"].float()
    exp = torch.where(w.unwrapped.reset_mask, torch.zeros_like(exp), exp)
    assert torch.equal(r, exp)
