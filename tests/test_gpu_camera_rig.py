"""GPU tests of camera rigs: several cameras per car, each rendered as its own view (the config's `cameras` list,
include/tinycarlo_b200.h tc_create_rig). View v = i*M + m is camera m of env i; observations are [N, M, ...].

The rig of most cases has M = 3 cameras: the config's camera, a rear camera (yaw 180) and a wider camera that sees twice as
far with its own per-env line thickness. Every frame is compared bit for bit with the oracle's frame of that view's camera row
at the car state (rig_util.oracle_views), after the buffer was poisoned with 0xAB, so that a skipped store shows."""
import contextlib
import os
import zlib

import numpy as np
import pytest
import torch

from hosttest_util import ht
from noise_util import reference_noise
from pair_util import make_config, oracle_env
from rig_util import REAR, oracle_view_segments, oracle_views
from test_gpu_map_shapes import LAUNCHES, decode, render_path
from test_gpu_parity import _check_segments
from tinycarlo_b200.camera_params import camera_row

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

M = 3
THICK2 = np.array([1, 2, 3, 5, 4], np.int32)   # camera 2's per-env thicknesses, cycled over the envs


def rig_config(fmt, res, cameras=None, map_name="knuffingen"):
    cfg = make_config(map_name, "rgb" if fmt == "rgb" else "classes", cam={"resolution": list(res)})
    mr = cfg["camera"]["max_range"]
    cfg["cameras"] = [{}, REAR, {"fov": 110, "max_range": 2 * mr}] if cameras is None else cameras
    return cfg


def plain_config(cfg):
    c = dict(cfg)
    c.pop("cameras")
    return c


@contextlib.contextmanager
def environ(setenv):
    old = {k: os.environ.get(k) for k in setenv}
    os.environ.update(setenv)
    try:
        yield
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)


def make_rig(cfg, n, fmt="classes", setenv=None, **kw):
    """the env, with camera 2's per-env thicknesses (the visible-set tables are rebuilt by set_camera_params, so the
    environment applies to both calls)"""
    from tinycarlo_b200 import TinyCarloVecEnv
    with environ(setenv or {}):
        env = TinyCarloVecEnv(cfg, n, device="cuda:0", obs_format=None if fmt in ("classes", "rgb") else fmt, **kw)
        if env.n_cameras == M:
            env.set_camera_params(camera=2, line_thickness=np.resize(THICK2, n))
    return env


def actions(rng, n, device="cuda:0"):
    """random commands, reverse included"""
    cc = np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
    man = rng.integers(0, 4, n).astype(np.int32)
    return cc, man, {"car_control": torch.from_numpy(cc).to(device), "maneuver": torch.from_numpy(man).to(device)}


def poison(env):
    env.obs.view(torch.uint8).fill_(0xAB)


def compare_views(env, sf, where, envs=None):
    """every view of the given envs (None: all) against the oracle's frame at state sf [N,8]; returns the frames compared"""
    fmt, H, W, Mn = env.observation_space_format, env.H, env.W, env.n_cameras
    idx = np.arange(env.num_envs) if envs is None else np.asarray(envs)
    if len(idx) == 0:
        return 0
    got = decode(env.obs[torch.from_numpy(idx).to(env.device)].flatten(0, 1), fmt, H, W)
    views = [int(i) * Mn + m for i in idx for m in range(Mn)]
    want = oracle_views(_omap(env), env._cam_rows, env._thickness, np.asarray(sf), Mn, H, W, "rgb" if fmt == "rgb" else "classes", views)[views]
    bad = np.nonzero((got != want).reshape(len(views), -1).any(axis=1))[0]
    if len(bad):
        v = views[int(bad[0])]
        pytest.fail(f"{where}: {len(bad)} of {len(views)} views differ from the oracle; first: env {v // Mn} camera {v % Mn} "
                    f"({int((got[bad[0]] != want[bad[0]]).sum())} values)")
    return len(views)


_OMAPS = {}


def _omap(env):
    from oracle import oracle as orc
    from tinycarlo_b200.config import resolve_map_path
    key = (resolve_map_path(env.config["map"], env.config_path), env.config["map"]["pixel_per_meter"])
    if key not in _OMAPS:
        _OMAPS[key] = orc.OracleMap(key[0], key[1])
    return _OMAPS[key]


def raw_views(env):
    """the frame buffer as bytes per env [N, M*frame bytes]"""
    return env.obs.view(torch.uint8).reshape(env.num_envs, -1).cpu().numpy()


# Camera 2's doubled reach makes Knuffingen's visible-set tables too large for 3 packed blocks per SM (tc_install_cull's rule),
# so the 84x84 rig takes the one-env kernel; the packed case's third camera looks sideways instead, at the shipped reach.
SIDE = [{}, REAR, {"orientation": [22, 0, 90]}]
# id: (obs format, resolution, envs, environment at construction, path tc_render_path takes[, cameras])
CASES = {
    "packed_84x84": ("classes", [84, 84], 64, {}, "packed", SIDE),
    "one_env_84x84": ("classes", [84, 84], 64, {"TC_ENV_PACK": "0"}, "one_env"),
    "per_class_u8_480x640": ("classes", [480, 640], 8, {}, "per_class"),
    "per_class_bf16_480x640": ("classes_bf16", [480, 640], 8, {}, "per_class"),
    "prims_bits_480x640": ("classes_bits", [480, 640], 8, {}, "prims"),
    "banded_rgb_480x640": ("rgb", [480, 640], 8, {}, "banded"),
    "unfused_segments_128x160": ("classes", [128, 160], 24, {}, "unfused"),
}


@pytest.mark.parametrize("case", list(CASES))
def test_rig_matches_oracle_on_every_render_path(case):
    """~30 steps of random commands (reverse included) with next-step autoreset and a masked reset halfway: every view
    of every step equals the oracle's frame for that view's camera row at the oracle env's state"""
    fmt, res, n, setenv, want_path, *cams = CASES[case]
    cfg = rig_config(fmt, res, *cams)
    env = make_rig(cfg, n, fmt, setenv, autoreset="next_step", debug_segments=want_path == "unfused")
    path = render_path(env)
    assert path == want_path, (case, path, env.render_info())
    assert env.obs.shape[:2] == (n, M)
    oenv = oracle_env(plain_config(cfg), n)
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    poison(env)
    env.reset(seed=zlib.crc32(case.encode()) & 0xFFFF)
    oenv.reset(env._spawn_nodes.cpu().numpy(), render=False)
    frames = compare_views(env, oenv.sf, "reset")
    done = np.zeros(n, bool)
    seg_stats = {"near": 0, "far": 0, "far_diff": 0}
    resets = 0
    for t in range(30):
        if t == 15:   # masked reset: the unselected envs' views keep the poison
            mask = rng.random(n) < 0.4
            mask[:2] = [True, False]
            poison(env)
            l0 = env.launch_count
            env.reset(mask=torch.from_numpy(mask))
            assert env.launch_count - l0 == LAUNCHES[want_path], "reset launches"
            oenv.reset(env._spawn_nodes.cpu().numpy(), mask=mask.astype(np.uint8), render=False)
            assert (raw_views(env)[~mask] == 0xAB).all(), "a masked reset wrote views of unselected envs"
            frames += compare_views(env, oenv.sf, "masked reset", envs=np.nonzero(mask)[0])
            done[mask] = False
        cc, man, act = actions(rng, n)
        poison(env)
        l0 = env.launch_count
        env.step(act)
        assert env.launch_count - l0 == LAUNCHES[want_path], (case, env.launch_count - l0)
        was = env.reset_mask.cpu().numpy()
        assert np.array_equal(was, done), t
        keep_sf, keep_si = oenv.sf.copy(), oenv.si.copy()
        oenv.step(cc.astype(np.float64), man, render=False)
        if was.any():   # next-step autoreset on the oracle: the finished envs are reset on the nodes the device drew
            oenv.sf[was], oenv.si[was] = keep_sf[was], keep_si[was]
            oenv.reset(env._spawn_nodes.cpu().numpy(), mask=was.astype(np.uint8), render=False)
            oenv.terminated[was] = 0
            oenv.truncated[was] = 0
            resets += int(was.sum())
        np.testing.assert_allclose(env.state_dict()["sf"].cpu().numpy()[:, :7], oenv.sf[:, :7], rtol=1e-9, atol=1e-11)
        frames += compare_views(env, oenv.sf, f"step {t}")
        if want_path == "unfused":
            cnt, seg = env.out["seg_count"].cpu().numpy(), env.out["seg_i32"].cpu().numpy()
            assert cnt.shape[0] == n * M
            off = env.map.ll_edge_off
            for v in range(n * M):
                ocnt, oseg = oracle_view_segments(_omap(env), env._cam_rows[v], env._thickness[v], oenv.sf[v // M], env.H, env.W)
                assert np.array_equal(cnt[v], ocnt), (t, v)
                for c in range(env.n_classes):
                    _check_segments(seg[v, off[c]:off[c] + cnt[v, c]], oseg[off[c]:off[c] + ocnt[c]], (case, t, v, c), seg_stats)
        done = (oenv.terminated | oenv.truncated).astype(bool)
    print(f"{case}: path {path}, {frames} views, {resets} autoresets, segments {seg_stats}")
    env.close()


def test_rig_changes_nothing_per_env():
    """a rig env and a rig-less env on the same config, seed and actions agree on every per-env output, and camera 0's
    views are the rig-less frames"""
    n = 256
    cfg = rig_config("classes", [128, 160])
    a = make_rig(cfg, n, autoreset="next_step")
    b = make_rig(plain_config(cfg), n, autoreset="next_step")
    a.reset(seed=3)
    b.reset(seed=3)
    assert torch.equal(a.obs[:, 0], b.obs)
    rng = np.random.default_rng(3)
    for t in range(25):
        if t == 12:
            mask = torch.from_numpy(rng.random(n) < 0.3)
            a.reset(mask=mask)
            b.reset(mask=mask)
        *_, act = actions(rng, n)
        oa, ob = a.step(act), b.step(act)
        for k in (1, 2, 3):
            assert torch.equal(oa[k], ob[k]), (t, k)
        assert oa[4].keys() == ob[4].keys()
        for k in ob[4]:
            assert torch.equal(oa[4][k], ob[4][k]), (t, k)
        assert torch.equal(a.reset_mask, b.reset_mask) and torch.equal(a.out["info_f64"], b.out["info_f64"])
        sa, sb = a.state_dict(), b.state_dict()
        assert torch.equal(sa["sf"], sb["sf"]) and torch.equal(sa["si"], sb["si"])
        assert torch.equal(a._spawn_nodes, b._spawn_nodes) and torch.equal(a._rng_state, b._rng_state)
        assert torch.equal(a.obs[:, 0], b.obs), t


@pytest.mark.parametrize("fmt,res", [("classes", [128, 160]), ("classes_bits", [480, 640])])
def test_rig_equals_a_flat_env_of_all_views(fmt, res):
    """a one-camera env of N*M envs with the rig's rows and each car's state M times renders the rig's views"""
    n = 48 if res[0] < 480 else 8
    cfg = rig_config(fmt, res)
    rig = make_rig(cfg, n, fmt, autoreset="next_step")
    rig.reset(seed=6)
    rng = np.random.default_rng(6)
    for _ in range(8):
        rig.step(actions(rng, n)[2])
    flat = make_rig(plain_config(cfg), n * M, fmt)
    flat.set_camera_rows(rig._cam_rows, line_thickness=rig._thickness)
    st = rig.state_dict()
    flat.load_state_dict({k: v.repeat_interleave(M, 0) for k, v in st.items()})
    assert render_path(flat) == render_path(rig)
    flat.render_obs()
    assert torch.equal(flat.obs, rig.obs.flatten(0, 1))
    stepped = rig.obs.clone()
    rig.render_obs()   # tc_render: the pose kernel's views
    assert torch.equal(rig.obs, stepped)


def test_single_camera_list_adds_the_axis():
    n = 32
    cfg = rig_config("classes", [84, 84], cameras=[{}])
    a, b = make_rig(cfg, n, autoreset="next_step"), make_rig(plain_config(cfg), n, autoreset="next_step")
    assert a.n_cameras == 1 and a.obs.shape == (n, 1, a.n_classes, 84, 84) and b.obs.shape == (n, a.n_classes, 84, 84)
    a.reset(seed=2)
    b.reset(seed=2)
    assert torch.equal(a.obs, b.obs[:, None])
    rng = np.random.default_rng(2)
    for _ in range(3):
        act = actions(rng, n)[2]
        a.step(act)
        b.step(act)
        assert torch.equal(a.obs, b.obs[:, None])


@pytest.mark.parametrize("res,n", [([84, 84], 64), ([480, 640], 8)])
def test_masked_reset_and_render_select_whole_envs(res, n):
    """tc_reset and tc_render with a per-env mask: the views of unselected envs keep the poison, those of selected envs equal
    the oracle; a selected env whose reset fails (no valid spawn node) is rendered at its old pose"""
    cfg = rig_config("classes", res)
    env = make_rig(cfg, n)
    env.reset(seed=8)
    rng = np.random.default_rng(8)
    for _ in range(3):
        env.step(actions(rng, n)[2])
    mask = rng.random(n) < 0.5
    mask[:3] = [True, False, True]
    nodes = env._spawn_nodes.cpu().numpy().copy()
    nodes[2] = -1   # env 2's reset fails
    old = env.state_dict()["sf"].cpu().numpy()
    poison(env)
    env.reset(mask=torch.from_numpy(mask), spawn_nodes=torch.from_numpy(nodes))
    sf = env.state_dict()["sf"].cpu().numpy()
    assert np.array_equal(sf[2], old[2])
    assert (raw_views(env)[~mask] == 0xAB).all()
    compare_views(env, sf, "masked reset", envs=np.nonzero(mask)[0])
    mask2 = ~mask
    poison(env)
    env.render_obs(mask=torch.from_numpy(mask2))
    assert (raw_views(env)[~mask2] == 0xAB).all()
    compare_views(env, sf, "masked render", envs=np.nonzero(mask2)[0])


def test_reach_covers_every_view():
    """the visible-set tables of the small-frame kernels are built for the farthest of all N*M cameras: here the last env's
    wide camera, which a loop over the first N rows would miss"""
    n = 64
    cfg = rig_config("classes", [84, 84], cameras=[{}, REAR, {"fov": 110}])
    env = make_rig(cfg, n)
    assert env.render_info()["block_per_env"] == 1
    far = 1.5 * cfg["camera"]["max_range"]   # (a reach that covers most of the map switches culling off: nothing to test)
    env.set_camera_params(camera=2, env_ids=[n - 1], max_range=far)
    H, W = env.H, env.W
    reach = [ht().ht_cull_radius_of(np.ascontiguousarray(r).ctypes.data, H, W) for r in env._cam_rows]
    assert min(reach) >= 0
    first_rows = max(reach[:n])
    assert max(reach) > first_rows, "the last env's camera 2 must see farther than the cameras of the first N rows"
    assert env.cull_info()["radius"] >= max(reach), (env.cull_info(), max(reach))
    env.reset(seed=5)
    rng = np.random.default_rng(5)
    frames = 0
    for t in range(6):
        frames += compare_views(env, env.state_dict()["sf"].cpu().numpy(), f"step {t}")
        env.step(actions(rng, n)[2])
    # the far camera does see beyond the nearer reach (otherwise the case would prove nothing)
    sf = env.state_dict()["sf"].cpu().numpy()
    row = env._cam_rows[(n - 1) * M + 2].copy()
    near = row.copy()
    near[16] = cfg["camera"]["max_range"]
    f_far = oracle_views(_omap(env), [row], [1], sf[n - 1:], 1, H, W, "classes")
    f_near = oracle_views(_omap(env), [near], [1], sf[n - 1:], 1, H, W, "classes")
    print(f"reach {max(reach):.3f} m, tables {env.cull_info()['radius']:.3f} m, first N rows {first_rows:.3f} m, {frames} views, "
          f"far camera differs from a near one: {bool((f_far != f_near).any())}")


def test_set_camera_params_per_camera():
    n = 32
    cfg = rig_config("classes", [84, 84])
    env = make_rig(cfg, n)
    env.reset(seed=4)
    before, rows0 = env.obs.clone(), env._cam_rows.copy()
    with pytest.raises(ValueError, match="rig"):
        env.set_camera_params(fov=90)
    for bad in (3, -1, [0, 5], 1.0, True):
        with pytest.raises(ValueError, match="camera"):
            env.set_camera_params(camera=bad, fov=90)
    fov = np.linspace(60, 120, n)
    env.set_camera_params(camera=1, fov=fov)
    rows = env._cam_rows
    cc = cfg["camera"]
    for i in range(n):
        assert np.array_equal(rows[i * M + 1], camera_row(cc["position"], REAR["orientation"], fov[i], cc["resolution"], cc["max_range"]))
    keep = np.arange(n * M) % M != 1
    assert np.array_equal(rows[keep], rows0[keep])
    poison(env)
    env.render_obs()
    assert torch.equal(env.obs[:, 0], before[:, 0]) and torch.equal(env.obs[:, 2], before[:, 2])
    assert not torch.equal(env.obs[:, 1], before[:, 1])
    compare_views(env, env.state_dict()["sf"].cpu().numpy(), "camera 1 changed")
    # camera lists and [N, M, 20] rows
    env.set_camera_params(camera=[0, 2], env_ids=[3], line_thickness=7)
    assert env._thickness[3 * M] == 7 and env._thickness[3 * M + 2] == 7 and env._thickness[3 * M + 1] == 2
    env.set_camera_rows(rows0.reshape(n, M, 20), line_thickness=np.full((n, M), 2))
    assert np.array_equal(env._cam_rows, rows0) and (env._thickness == 2).all()


def test_noise_wrapper_on_rig_views():
    """camera 0's views get the rig-less noise; views of camera m > 0 the noise of counter word 3 = m"""
    from tinycarlo_b200 import TinyCarloVecEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    n, off, seed, n_blobs, max_radius = 24, 100, 0x5EED1234AB, 5, 20
    cfg = rig_config("classes", [84, 84])
    rig, clean = make_rig(cfg, n, env_index_offset=off), make_rig(cfg, n, env_index_offset=off)
    plain = TinyCarloVecEnv(plain_config(cfg), n, device="cuda:0", env_index_offset=off)
    wr = NoiseObservationWrapper(rig, blob_max_radius=max_radius, n_blobs=n_blobs, seed=seed)
    wp = NoiseObservationWrapper(plain, blob_max_radius=max_radius, n_blobs=n_blobs, seed=seed)
    for e in (wr, wp, clean):
        e.reset(seed=1)
    rng = np.random.default_rng(1)
    for t in range(3):
        act = actions(rng, n)[2]
        o_r, o_p, o_c = wr.step(act)[0], wp.step(act)[0], clean.step(act)[0]
        assert torch.equal(o_r[:, 0], o_p), t
        got, c = o_r.cpu().numpy(), o_c.cpu().numpy()
        changed = 0
        for i in range(n):
            for m in range(1, M):
                want = reference_noise(c[i, m].copy(), off + i, m, seed, t, n_blobs, max_radius)
                assert np.array_equal(got[i, m], want), (t, i, m)
                changed += int((want != c[i, m]).any())
        assert changed > 0


def test_graph_checkpoint_and_host_step():
    n = 128
    cfg = rig_config("classes", [84, 84])
    eager, graphed = make_rig(cfg, n, autoreset="next_step"), make_rig(cfg, n, autoreset="next_step")
    rng = np.random.default_rng(11)
    slot = {k: v.clone() for k, v in actions(rng, n)[2].items()}
    for e in (eager, graphed):
        e.reset(seed=21)
    for _ in range(3):   # capture()'s warm-up steps
        eager.step(slot)
    g = graphed.capture(lambda e: slot, steps=5, warmup=3)
    for r in range(4):
        for k, v in actions(rng, n)[2].items():
            slot[k].copy_(v)
        for _ in range(5):
            eager.step(slot)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(eager.obs, graphed.obs), r
        assert torch.equal(eager.state_dict()["sf"], graphed.state_dict()["sf"]), r
    # checkpoint / restore re-renders all views
    ck = eager.checkpoint()
    want = eager.obs.clone()
    eager.step(slot)
    assert not torch.equal(eager.obs, want)
    eager.restore(ck)
    assert torch.equal(eager.obs, want)
    # step_host with obs_host carries all views in one copy
    cc, man, act = actions(rng, n)
    graphed.restore(ck)
    graphed.step(act)
    reward, term, trunc = torch.zeros(n), torch.zeros(n, dtype=torch.uint8), torch.zeros(n, dtype=torch.uint8)
    obs_host = torch.empty(eager.obs.shape, dtype=eager.obs.dtype).pin_memory()
    eager.step_host(torch.from_numpy(cc), torch.from_numpy(man), reward, term, trunc, obs_host=obs_host)
    assert obs_host.shape == (n, M, eager.n_classes, 84, 84)
    assert torch.equal(obs_host, graphed.obs.cpu()) and torch.equal(obs_host, eager.obs.cpu())
    assert torch.equal(reward, graphed.out["reward"].cpu())


def test_grouped_and_single_env_with_a_rig():
    from tinycarlo_b200 import TinyCarloEnv, TinyCarloGroupedVecEnv
    cfg = rig_config("classes", [84, 84])
    ge = TinyCarloGroupedVecEnv(cfg, [(40, [84, 84]), (24, [64, 96])], device="cuda:0", autoreset="next_step")
    obs, _ = ge.reset(seed=1)
    C_ = ge.envs[0].n_classes
    assert [tuple(o.shape) for o in obs] == [(40, M, C_, 84, 84), (24, M, C_, 64, 96)]
    with pytest.raises(ValueError, match="rig"):
        ge.set_camera_params(fov=90)
    fov = np.linspace(70, 100, 64)
    ge.set_camera_params(camera=1, fov=fov)
    rng = np.random.default_rng(3)
    for _ in range(2):
        ge.step(actions(rng, 64)[2])
    for e, (a, b) in zip(ge.envs, [(0, 40), (40, 64)]):
        cc = cfg["camera"]
        assert np.array_equal(e._cam_rows[1::M], np.stack([camera_row(cc["position"], REAR["orientation"], f, [e.H, e.W], cc["max_range"])
                                                           for f in fov[a:b]]))
        compare_views(e, e.state_dict()["sf"].cpu().numpy(), f"group {e.H}x{e.W}", envs=range(0, e.num_envs, 5))
    # the single env: camera 0 is the reference's camera, `cameras` holds one facade per camera
    se = TinyCarloEnv(config=cfg, device="cuda:0")
    assert se.observation_space.shape == (M, C_, 84, 84) and len(se.cameras) == M and se.camera is se.cameras[0]
    obs, _ = se.reset(seed=0)
    assert obs.shape == (M, C_, 84, 84)
    obs = se.step({"car_control": [-0.5, 0.2], "maneuver": 0})[0]
    assert np.array_equal(obs, se._vec.obs[0].cpu().numpy())
    rows0 = se._vec._cam_rows.copy()
    se.camera.fov = 100
    se.camera.update_params()
    rows = se._vec._cam_rows
    assert not np.array_equal(rows[0], rows0[0]) and np.array_equal(rows[1:], rows0[1:])
    assert np.array_equal(se.camera.E, rows[0, :12].reshape(3, 4))
    se.cameras[2].max_range = 0.7
    se.cameras[2].update_params()
    assert rows[2, 16] == 0.7 and np.array_equal(rows[1], rows0[1])
    assert np.array_equal(se.cameras[1].E, rows0[1, :12].reshape(3, 4))
    obs = se.step({"car_control": [0.5, 0.0], "maneuver": 0})[0]
    assert np.array_equal(se.cameras[1].get_last_frame_classes(), obs[1])
    compare_views(se._vec, se._vec.state_dict()["sf"].cpu().numpy(), "single env")
    se.render_mode = "rgb_array"
    frame = se.render()
    assert frame.shape == (84, 84, 3) and np.array_equal(frame, se._vec.render_rgb()[0, 0].cpu().numpy())
