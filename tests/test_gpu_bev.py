"""The bird's-eye view on the device (config section `bev`, tc_bev_kernel) against the numpy + cv2 restatement of its
contract (tests/bev_util.py), and what switching it on must leave alone."""
import numpy as np
import pytest
import torch

from bev_util import oracle_bev_ulp, pack_bits
from tinycarlo_b200 import TinyCarloVecEnv
from tinycarlo_b200.config import make_config

pytestmark = pytest.mark.gpu

BEV = {"resolution": [128, 128], "pixel_per_meter": 128, "line_thickness": 2, "route": True}


def bev_config(map_name, fmt="classes", bev=None, cam=None):
    cfg = make_config(map_name, fmt, cam=cam)
    if bev is not None:
        cfg["bev"] = dict(bev)
    return cfg


def actions(rng, n, t, dev):
    """random commands, mostly forward, with maneuvers that switch every few steps"""
    cc = np.stack([rng.uniform(-0.3, 1.0, n), rng.uniform(-1.0, 1.0, n)], 1).astype(np.float32)
    man = ((np.arange(n) + t // 4) % 4).astype(np.int32) if t % 4 == 0 else (np.arange(n) % 4).astype(np.int32)
    man[rng.random(n) < 0.3] = rng.integers(0, 4)
    return {"car_control": torch.from_numpy(cc).to(dev), "maneuver": torch.from_numpy(man).to(dev)}


def check_frames(env, envs=None):
    """env.bev against the oracle fed with the device state -> (frames compared, frames that needed the one-ulp cos/sin nudge);
    fails on any other difference"""
    st = env.state_dict()
    sf, si = st["sf"].cpu().numpy(), st["si"].cpu().numpy()
    got = env.bev.cpu().numpy()
    H, W = env.bev_cfg["resolution"]
    kw = dict(H=H, W=W, pixel_per_meter=env.bev_cfg["pixel_per_meter"], car_pixel=env.bev_cfg["car_pixel"],
              thickness=env.bev_cfg["line_thickness"], route=env.bev_cfg["route"])
    nudged = 0
    ids = range(env.num_envs) if envs is None else envs
    for i in ids:
        r = oracle_bev_ulp(env.map, sf[i], si[i], got[i], **kw)
        assert r >= 0, f"env {i}: BEV differs from the oracle (state {sf[i][:3]})"
        nudged += r
    return len(ids), nudged


@pytest.mark.parametrize("map_name", ["knuffingen", "simple_layout"])
def test_bev_rollout_matches_oracle(map_name):
    n, steps = 2048, 30
    env = TinyCarloVecEnv(bev_config(map_name, bev=BEV), n, device="cuda:0", autoreset="next_step")
    rng = np.random.default_rng(7)
    env.reset(seed=3)
    frames, nudged = check_frames(env)
    drawn = 0
    for t in range(steps):
        _, _, _, _, info = env.step(actions(rng, n, t, env.device))
        assert info["bev"] is env.bev
        f, u = check_frames(env)
        frames += f
        nudged += u
        drawn += int(env.bev.flatten(1).any(1).sum().item())
    print(f"{map_name}: {frames} BEV frames equal to the oracle, {nudged} of them with cos/sin moved by one ulp")
    assert drawn > steps * n // 2   # the lanes are in view


def test_bev_bits_is_u8_packed():
    n = 512
    envs = [TinyCarloVecEnv(bev_config("knuffingen", bev=dict(BEV, format=f)), n, device="cuda:0", autoreset="next_step")
            for f in ("classes", "classes_bits")]
    assert envs[1].bev.dtype == torch.int32 and tuple(envs[1].bev.shape) == (n, 6, 128 * 128 // 32)
    rng = np.random.default_rng(1)
    for e in envs:
        e.reset(seed=5)
    for t in range(8):
        a = actions(rng, n, t, envs[0].device)
        for e in envs:
            e.step(a)
        assert np.array_equal(pack_bits(envs[0].bev.cpu().numpy()), envs[1].bev.cpu().numpy())


def test_bev_changes_nothing_else():
    n = 1024
    envs = [TinyCarloVecEnv(bev_config("knuffingen", bev=b), n, device="cuda:0", autoreset="next_step") for b in (None, BEV)]
    assert envs[0].bev is None and "bev" not in envs[0].reset(seed=9)[1]
    envs[1].reset(seed=9)
    rng = np.random.default_rng(2)
    l0 = [e.launch_count for e in envs]
    for t in range(10):
        a = actions(rng, n, t, envs[0].device)
        outs = [e.step(a) for e in envs]
        assert torch.equal(outs[0][0], outs[1][0])
        for k in (1, 2, 3):
            assert torch.equal(outs[0][k], outs[1][k])
        assert set(outs[1][4]) == set(outs[0][4]) | {"bev"}
        for k, v in outs[0][4].items():
            assert torch.equal(v, outs[1][4][k]), k
        for k, v in envs[0].out.items():
            assert torch.equal(v, envs[1].out[k]), k
    assert envs[1].launch_count - l0[1] == envs[0].launch_count - l0[0] + 10   # one launch more per step


def test_bev_masked_reset_and_no_observation():
    n = 256
    env = TinyCarloVecEnv(bev_config("simple_layout", bev=BEV), n, device="cuda:0")
    env.reset(seed=4)
    env.bev.fill_(77)
    mask = torch.zeros(n, dtype=torch.bool, device=env.device)
    mask[::3] = True
    env.reset(mask=mask)
    b = env.bev.cpu().numpy()
    m = mask.cpu().numpy()
    assert np.all(b[~m] == 77)
    assert np.all((b[m] == 0) | (b[m] == 255))
    check_frames(env, envs=np.nonzero(m)[0][:64])
    # the camera switch does not touch the BEV: it is drawn on every step
    env.no_observation = True
    env.bev.fill_(77)
    env.step(actions(np.random.default_rng(0), n, 0, env.device))
    assert not (env.bev == 77).any()
    check_frames(env, envs=range(0, n, 5))
    env.bev.fill_(77)
    env.render_bev(mask=mask)
    b = env.bev.cpu().numpy()
    assert np.all(b[~m] == 77) and np.all((b[m] == 0) | (b[m] == 255))


def test_bev_graph_and_checkpoint():
    n = 1024
    cfg = bev_config("knuffingen", bev=BEV)
    eager, graphed = (TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step") for _ in range(2))
    rng = np.random.default_rng(11)
    acts = [actions(rng, n, t, eager.device) for t in range(6)]
    slot = {k: v.clone() for k, v in acts[0].items()}
    for e in (eager, graphed):
        e.reset(seed=21)
    # capture() runs its warm-up steps (3) with the slot's action before the graph: replay the same on the eager env
    for _ in range(3):
        eager.step(slot)
    g = graphed.capture(lambda e: slot, steps=1, warmup=3)
    for a in acts:
        eager.step(a)
        for k in slot:
            slot[k].copy_(a[k])
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(eager.bev, graphed.bev)
        assert torch.equal(eager.obs, graphed.obs)
    ck = eager.checkpoint()
    want = eager.bev.clone()
    eager.step(acts[0])
    assert not torch.equal(eager.bev, want)
    eager.restore(ck)
    assert torch.equal(eager.bev, want)


def test_bev_grouped_and_single_env():
    from tinycarlo_b200 import TinyCarloEnv, TinyCarloGroupedVecEnv
    cfg = bev_config("simple_layout", bev=BEV)
    ge = TinyCarloGroupedVecEnv(cfg, [(100, [84, 84]), (60, [64, 96])], device="cuda:0", autoreset="next_step")
    _, info = ge.reset(seed=1)
    assert tuple(info["bev"].shape) == (160, 6, 128, 128)
    rng = np.random.default_rng(5)
    for t in range(3):
        *_, info = ge.step(actions(rng, 160, t, ge.device))
        assert torch.equal(info["bev"], torch.cat([e.bev for e in ge.envs]))
    for e in ge.envs:
        check_frames(e, envs=range(0, e.num_envs, 7))
    se = TinyCarloEnv(config=cfg, device="cuda:0")
    _, info = se.reset(seed=0)
    assert isinstance(info["bev"], np.ndarray) and info["bev"].shape == (6, 128, 128)
    *_, info = se.step({"car_control": [0.5, 0.1], "maneuver": 0})
    assert np.array_equal(info["bev"], se._vec.bev[0].cpu().numpy())
    check_frames(se._vec)
    plain = TinyCarloEnv(config=make_config("simple_layout", "classes"), device="cuda:0")
    assert "bev" not in plain.reset(seed=0)[1]
    assert "bev" not in plain.step({"car_control": [0.5, 0.1], "maneuver": 0})[4]


def test_bev_headline_size():
    n = 16384
    env = TinyCarloVecEnv(bev_config("knuffingen", bev={"resolution": [128, 128]}, cam={"resolution": [480, 640]}), n, device="cuda:0",
                          autoreset="next_step")
    env.reset(seed=8)
    env.step(actions(np.random.default_rng(3), n, 0, env.device))
    ids = np.random.default_rng(4).choice(n, 256, replace=False)
    frames, nudged = check_frames(env, envs=ids)
    print(f"headline size: {frames} sampled BEV frames equal to the oracle, {nudged} with cos/sin moved by one ulp")
