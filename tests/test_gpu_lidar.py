"""The range scan on the device (config section `lidar`, tc_lidar_kernel) against the numpy restatement of its contract
(tests/lidar_util.py), float32 bit pattern for bit pattern, and what switching it on must leave alone: rollouts with
autoresets and masked resets, the synthetic edge cases, a class larger than one shared-memory tile, 1 / 4099 / 16384 envs,
guard bands and determinism, every entry point that launches the kernel, a camera rig, the grouped and the single env."""
import ctypes as C

import numpy as np
import pytest
import torch

import map_shapes_util as M
from lidar_util import SYN_LAYERS, SYN_RANGE, oracle_lidar_ulp, synthetic_map
from rig_util import REAR
from tinycarlo_b200 import TinyCarloVecEnv, _lib
from tinycarlo_b200.config import make_config

pytestmark = pytest.mark.gpu

LIDAR = {"rays": 64, "fov": 360, "max_range": 0.5}


def lidar_config(map_name, lidar=None, cam=None, tmp_path=None):
    cfg = make_config("knuffingen" if map_name in M.MAPS else map_name, "classes", cam=cam)
    if map_name in M.MAPS:
        cfg["map"] = {"json_path": M.write(M.MAPS[map_name](), tmp_path, map_name), "pixel_per_meter": M.PPM,
                      "spawn_points": list(M.SPAWN_KNUFF)}
    if lidar is not None:
        cfg["lidar"] = dict(lidar)
    return cfg


def actions(rng, n, t, dev):
    cc = np.stack([rng.uniform(-0.3, 1.0, n), rng.uniform(-1.0, 1.0, n)], 1).astype(np.float32)
    man = ((np.arange(n) + t // 4) % 4).astype(np.int32)
    man[rng.random(n) < 0.3] = rng.integers(0, 4)
    return {"car_control": torch.from_numpy(cc).to(dev), "maneuver": torch.from_numpy(man).to(dev)}


def check_scans(env, envs=None):
    """env.lidar against the oracle fed with the device state -> counts [scans compared, scans that needed the one-ulp cos/sin
    nudge, those of them whose car sits exactly on a lanepath node]; fails on any other difference (-0.0 against +0.0
    included)"""
    sf = env.state_dict()["sf"].cpu().numpy()
    got = env.lidar.cpu().numpy()
    li = env.lidar_cfg
    kw = dict(rays=li["rays"], fov=li["fov"], max_range=li["max_range"], origin=li["origin"])
    counts = np.zeros(3, np.int64)
    for i in (range(env.num_envs) if envs is None else envs):
        r = oracle_lidar_ulp(env.map, sf[i], got[i], **kw)
        assert r >= 0, f"env {i}: scan differs from the oracle (state {sf[i][:3]})"
        on_node = bool((env.map.lp_nodes == sf[i, :2]).all(1).any())
        counts += (1, r, r * on_node)
    return counts


def report(what, counts):
    """prints the counts; fails when more than 0.1 % of the scans of cars off the lanepath nodes needed the nudge (the BEV's rule)"""
    scans, nudged, on_node = (int(v) for v in counts)
    print(f"{what}: {scans} scans equal to the oracle, {nudged} of them with cos/sin moved by one ulp ({on_node} with the car on a "
          f"lanepath node)")
    assert (nudged - on_node) * 1000 <= scans, f"{what}: {nudged - on_node} of {scans} scans off the lanepath nodes needed the nudge"


def poison(env):
    env.lidar.view(torch.int32).fill_(0x7FABCDEF)


def poisoned(env):
    return (env.lidar.view(torch.int32).flatten(1) == 0x7FABCDEF).all(1).cpu().numpy()


@pytest.mark.parametrize("map_name", ["knuffingen", "simple_layout"])
def test_lidar_rollout_matches_oracle(map_name):
    """reset, 10 steps with next-step autoresets (a quarter of the envs marked done at step 3), a masked reset"""
    n, steps = 512, 10
    env = TinyCarloVecEnv(lidar_config(map_name, LIDAR), n, device="cuda:0", autoreset="next_step")
    assert tuple(env.lidar.shape) == (n, env.n_classes, 64) and env.lidar.dtype == torch.float32
    rng = np.random.default_rng(7)
    poison(env)
    env.reset(seed=3)
    counts = check_scans(env)
    hits = autoresets = 0
    for t in range(steps):
        if t == 3:
            env.mark_done(torch.from_numpy(np.arange(n) % 4 == 0).to(env.device))
        poison(env)
        *_, info = env.step(actions(rng, n, t, env.device))
        assert info["lidar"] is env.lidar
        autoresets += int(env.reset_mask.sum().item())
        counts += check_scans(env)
        hits += int((env.lidar < 0.5).flatten(1).any(1).sum().item())
    mask = rng.random(n) < 0.5
    poison(env)
    env.reset(mask=torch.from_numpy(mask))
    assert poisoned(env)[~mask].all() and not poisoned(env)[mask].any()
    counts += check_scans(env, envs=np.nonzero(mask)[0])
    report(map_name, counts)
    assert autoresets >= n // 4 and hits > steps * n // 2


@pytest.mark.parametrize("rays,fov", [(1, 360.0), (3, 1e-3), (65, 90.0), (1023, 360.0)])
def test_lidar_synthetic_edge_cases(rays, fov, tmp_path):
    """the host test's synthetic cases on the device at θ = 0 (device cos(0) = 1, sin(0) = 0 exactly): u = 0 and 1, t = +0.0,
    parallel / collinear / zero-length edges, max_range and one ulp beyond it, an edge crossing the cull's square, u an ulp either
    side of 1"""
    cfg = make_config("knuffingen", "classes", cam={"resolution": [64, 64]})
    cfg["map"] = {"json_path": synthetic_map(tmp_path), "pixel_per_meter": 1, "spawn_points": [0]}
    cfg["lidar"] = {"rays": rays, "fov": fov, "max_range": SYN_RANGE}
    env = TinyCarloVecEnv(cfg, 2, device="cuda:0")
    env.reset(seed=0)
    sf = np.zeros((2, 8))
    sf[1, :3] = [-0.05, 0.0, 0.0]
    env.load_state_dict({"sf": torch.from_numpy(sf), "si": torch.full((2, 16), -1, dtype=torch.int32)})
    poison(env)
    env.render_lidar()
    assert check_scans(env)[1] == 0
    got = env.lidar.cpu().numpy()
    j = (rays - 1) // 2
    fwd = {name: got[0, p, j] for p, name in enumerate(SYN_LAYERS)}
    assert fwd["zero"] == 0.0 and not np.signbit(fwd["zero"])
    assert not np.signbit(got).any()
    for name in ("parallel", "collinear", "point", "at_range", "beyond", "near1_2", "near1_3"):
        assert fwd[name] == np.float32(SYN_RANGE), name
    assert fwd["u0"] == np.float32(0.2) and fwd["u1"] == np.float32(0.15) and fwd["crossing"] == np.float32(0.1)
    assert fwd["near1_-2"] == fwd["near1_-3"] == np.float32(0.12)


@pytest.mark.parametrize("case", ["K1_1024", "K16_300", "knuff_1", "n1", "n4099", "n16384"])
def test_lidar_shapes_and_env_counts(case, tmp_path):
    """K1 holds all 739 of Knuffingen's edges in one class (three tiles of 256 at 1024 rays, twelve of 64 at 64 rays); 16 classes
    at 300 rays (two rays for some threads); one ray; 1, 4099 and 16384 envs (sampled at 16384)"""
    map_name, lidar, n = {"K1_1024": ("K1", dict(LIDAR, rays=1024, max_range=3.0), 64),
                          "K16_300": ("K16", dict(LIDAR, rays=300, fov=270, origin=[0.02, -0.01]), 64),
                          "knuff_1": ("knuffingen", dict(LIDAR, rays=1, fov=30), 64),
                          "n1": ("knuffingen", LIDAR, 1), "n4099": ("knuffingen", dict(LIDAR, rays=33), 4099),
                          "n16384": ("knuffingen", LIDAR, 16384)}[case]
    env = TinyCarloVecEnv(lidar_config(map_name, lidar, cam={"resolution": [64, 64]}, tmp_path=tmp_path), n, device="cuda:0",
                          autoreset="next_step")
    rng = np.random.default_rng(len(case))
    ids = None if n <= 4099 else rng.choice(n, 512, replace=False)
    if n == 4099:
        ids = np.r_[0:64, n - 64:n, rng.choice(n, 256, replace=False)]
    poison(env)
    env.reset(seed=2)
    assert not poisoned(env).any()
    counts = check_scans(env, ids)
    for t in range(3):
        poison(env)
        env.step(actions(rng, n, t, env.device))
        assert not poisoned(env).any()
        counts += check_scans(env, ids)
    report(case, counts)


def test_lidar_guard_bands_determinism_and_state_error():
    """tc_set_lidar pointed at a payload inside [guard | payload | guard] (one float past a 16-byte boundary): the sentinels
    survive, every float of the poisoned payload is rewritten, six repeats of a step from the same state give identical scans;
    tc_render_lidar without a scan set is TC_ERR_STATE"""
    n = 37
    env = TinyCarloVecEnv(lidar_config("knuffingen", dict(LIDAR, rays=100)), n, device="cuda:0")
    G, off = 4096, 4
    nb = env.lidar.numel() * 4
    buf = torch.full((G + off + nb + G,), 0x5C, dtype=torch.uint8, device=env.device)
    env.lidar = buf[G + off:G + off + nb].view(torch.float32).view(env.lidar.shape)
    li = env.lidar_cfg
    d = _lib.TcLidarDesc(li["rays"], li["fov"], li["max_range"], *li["origin"])
    _lib.check(env._L.tc_set_lidar(env._h, C.byref(d), C.c_void_p(env.lidar.data_ptr())), "tc_set_lidar")

    def guards_intact():
        g = buf.cpu().numpy()
        return (g[:G + off] == 0x5C).all() and (g[G + off + nb:] == 0x5C).all()
    rng = np.random.default_rng(17)
    env.reset(seed=6)
    counts = np.zeros(3, np.int64)
    for t in range(3):
        a = actions(rng, n, t, env.device)
        st0 = {k: v.clone() for k, v in env.state_dict().items()}
        first = None
        for rep in range(6):
            env.load_state_dict(st0)
            poison(env)
            env.step(a)
            assert not (env.lidar.view(torch.int32) == 0x7FABCDEF).any()
            if first is None:
                first = env.lidar.clone()
                counts += check_scans(env)
            else:
                assert torch.equal(env.lidar.view(torch.int32), first.view(torch.int32)), f"step {t}, repetition {rep}"
        assert guards_intact(), f"step {t}: a guard band was overwritten"
    report("guard bands", counts)
    assert env._L.tc_set_lidar(env._h, None, None) == 0
    assert env._L.tc_render_lidar(env._h, None, None) == -4   # TC_ERR_STATE
    assert b"no scan set" in env._L.tc_last_error()


def test_lidar_changes_nothing_else_and_launch_counts():
    """with the scan on, obs, info, BEV, rewards and flags equal the run without it, one launch more per step; without the section
    nothing changes; with no_observation a step launches the tracking kernel and the scan only"""
    n = 1024
    bev = {"resolution": [64, 64], "route": True}
    base = lidar_config("knuffingen")
    base["bev"] = bev
    envs = [TinyCarloVecEnv(dict(base, **extra), n, device="cuda:0", autoreset="next_step") for extra in ({}, {"lidar": LIDAR})]
    assert envs[0].lidar is None and "lidar" not in envs[0].reset(seed=9)[1]
    envs[1].reset(seed=9)
    rng = np.random.default_rng(2)
    l0 = [e.launch_count for e in envs]
    for t in range(8):
        a = actions(rng, n, t, envs[0].device)
        outs = [e.step(a) for e in envs]
        assert torch.equal(outs[0][0], outs[1][0])
        for k in (1, 2, 3):
            assert torch.equal(outs[0][k], outs[1][k])
        assert set(outs[1][4]) == set(outs[0][4]) | {"lidar"}
        for k, v in outs[0][4].items():
            assert torch.equal(v, outs[1][4][k]), k
        for k, v in envs[0].out.items():
            assert torch.equal(v, envs[1].out[k]), k
    assert envs[1].launch_count - l0[1] == envs[0].launch_count - l0[0] + 8
    # no_observation: tracking + scan, one launch more than tracking alone
    plain, scan = (TinyCarloVecEnv(lidar_config("knuffingen", li), n, device="cuda:0", autoreset="next_step") for li in (None, LIDAR))
    per_step = []
    for e in (plain, scan):
        e.reset(seed=1)
        e.no_observation = True
        c0 = e.launch_count
        for t in range(5):
            e.step(actions(rng, n, t, e.device))
        per_step.append((e.launch_count - c0) / 5)
    assert per_step == [1, 2], per_step
    report("no_observation", check_scans(scan, envs=range(0, n, 4)))


def test_lidar_step_f64_step_host_restore_and_graph():
    """the scan after tc_step_f64, tc_step_host and restore equals the oracle; a captured graph replays what eager stepping gives"""
    n = 256
    cfg = lidar_config("knuffingen", dict(LIDAR, rays=48, fov=200, origin=[0.03, 0.01]), cam={"resolution": [64, 64]})
    env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    rng = np.random.default_rng(12)
    env.reset(seed=12)
    counts = check_scans(env)
    for t in range(3):
        a = actions(rng, n, t, env.device)
        a["car_control"] = a["car_control"].double()
        poison(env)
        env.step(a)
        counts += check_scans(env)
    reward, term, trunc = torch.zeros(n), torch.zeros(n, dtype=torch.uint8), torch.zeros(n, dtype=torch.uint8)
    for t in range(3):
        a = actions(rng, n, t, env.device)
        poison(env)
        env.step_host(a["car_control"].cpu(), a["maneuver"].cpu(), reward, term, trunc)
        counts += check_scans(env)
    ck = env.checkpoint()
    want = env.lidar.clone()
    env.step(actions(rng, n, 0, env.device))
    assert not torch.equal(env.lidar, want)
    poison(env)
    env.restore(ck)
    assert torch.equal(env.lidar, want)
    report("tc_step_f64, tc_step_host, restore", counts)

    eager, graphed = (TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step") for _ in range(2))
    acts = [actions(rng, n, t, eager.device) for t in range(6)]
    slot = {k: v.clone() for k, v in acts[0].items()}
    for e in (eager, graphed):
        e.reset(seed=21)
    for _ in range(3):
        eager.step(slot)
    g = graphed.capture(lambda e: slot, steps=1, warmup=3)
    for a in acts:
        eager.step(a)
        for k in slot:
            slot[k].copy_(a[k])
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(eager.lidar, graphed.lidar)
        assert torch.equal(eager.obs, graphed.obs)


def test_lidar_on_a_rig_grouped_and_single_env():
    """a camera rig (M = 3) gives the scan of the one-camera env, env for env, and its masked reset / render select envs, not
    views; the grouped env concatenates info["lidar"]; the single env returns it as numpy [C, R]"""
    from tinycarlo_b200 import TinyCarloEnv, TinyCarloGroupedVecEnv
    n = 64
    plain = lidar_config("knuffingen", LIDAR, cam={"resolution": [64, 64]})
    rig = dict(plain, cameras=[{}, REAR, {"fov": 110}])
    envs = [TinyCarloVecEnv(c, n, device="cuda:0", autoreset="next_step") for c in (rig, plain)]
    assert envs[0].n_cameras == 3 and tuple(envs[0].lidar.shape) == (n, 5, 64)
    rng = np.random.default_rng(3)
    for e in envs:
        e.reset(seed=3)
    assert torch.equal(envs[0].lidar, envs[1].lidar)
    for t in range(4):
        a = actions(rng, n, t, envs[0].device)
        for e in envs:
            e.step(a)
        assert torch.equal(envs[0].lidar, envs[1].lidar), f"step {t}"
    env = envs[0]
    mask = rng.random(n) < 0.5
    mask[:4] = [True, False, True, False]
    poison(env)
    env.reset(mask=torch.from_numpy(mask))
    assert poisoned(env)[~mask].all() and not poisoned(env)[mask].any()
    counts = check_scans(env, envs=np.nonzero(mask)[0])
    poison(env)
    env.render_lidar(mask=torch.from_numpy(~mask))
    assert poisoned(env)[mask].all() and not poisoned(env)[~mask].any()
    counts += check_scans(env, envs=np.nonzero(~mask)[0])
    report("rig", counts)

    cfg = lidar_config("simple_layout", LIDAR)
    ge = TinyCarloGroupedVecEnv(cfg, [(100, [84, 84]), (60, [64, 96])], device="cuda:0", autoreset="next_step")
    _, info = ge.reset(seed=1)
    assert tuple(info["lidar"].shape) == (160, 5, 64)
    for t in range(3):
        *_, info = ge.step(actions(rng, 160, t, ge.device))
        assert torch.equal(info["lidar"], torch.cat([e.lidar for e in ge.envs]))
    for e in ge.envs:
        check_scans(e, envs=range(0, e.num_envs, 7))
    se = TinyCarloEnv(config=cfg, device="cuda:0")
    _, info = se.reset(seed=0)
    assert isinstance(info["lidar"], np.ndarray) and info["lidar"].shape == (5, 64) and info["lidar"].dtype == np.float32
    *_, info = se.step({"car_control": [0.5, 0.1], "maneuver": 0})
    assert np.array_equal(info["lidar"], se._vec.lidar[0].cpu().numpy())
    check_scans(se._vec)
    plain_se = TinyCarloEnv(config=make_config("simple_layout", "classes"), device="cuda:0")
    assert "lidar" not in plain_se.reset(seed=0)[1]
