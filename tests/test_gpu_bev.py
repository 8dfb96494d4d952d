"""The bird's-eye view on the device (config section `bev`, tc_bev_kernel) against the numpy + cv2 restatement of its
contract (tests/bev_util.py), and what switching it on must leave alone.

Beyond the 128x128 default: a table of geometries (every thickness, frames whose planes do not start on a word and whose env
bases are not 16-byte aligned, extreme aspect ratios, 1 to 16 planes, scales from 2 to 1e9 px/m, car pixels in and far outside
the frame, the bit-packed format, the largest frames the 200 KB stacked plane accepts), placed poses at the culling margin of
tc_bev_segment, guard bands / full overwrite / determinism, and every entry point that launches the kernel (tc_step_f64,
tc_step_host, restore, masked tc_reset and tc_render_bev on a camera rig)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import map_shapes_util as M
from bev_util import oracle_bev_ulp, pack_bits
from rig_util import REAR
from tinycarlo_b200 import TinyCarloVecEnv, _lib
from tinycarlo_b200.config import BEV_SMEM_MAX, MAPS_DIR, PPM, bev_params, make_config
from tinycarlo_b200.maptables import MapTables

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

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
    """env.bev against the oracle fed with the device state -> counts [frames compared, frames that needed the one-ulp cos/sin
    nudge, those of them whose car sits exactly on a lanepath node]; fails on any other difference.
    A car on a lanepath node (a spawn pose, or a car that has not moved since) heads along a lanepath edge: the map points on
    that line have a lateral offset that is zero in exact arithmetic, and the last bit of cos/sin decides on which side of the
    car pixel's column they are truncated. About a quarter of Knuffingen's spawn poses are that sensitive; other poses almost
    never are."""
    st = env.state_dict()
    sf, si = st["sf"].cpu().numpy(), st["si"].cpu().numpy()
    got = env.bev.cpu().numpy()
    H, W = env.bev_cfg["resolution"]
    kw = dict(H=H, W=W, pixel_per_meter=env.bev_cfg["pixel_per_meter"], car_pixel=env.bev_cfg["car_pixel"],
              thickness=env.bev_cfg["line_thickness"], route=env.bev_cfg["route"], bits=env.bev_cfg["format"] == "classes_bits")
    counts = np.zeros(3, np.int64)
    ids = range(env.num_envs) if envs is None else envs
    for i in ids:
        r = oracle_bev_ulp(env.map, sf[i], si[i], got[i], **kw)
        assert r >= 0, f"env {i}: BEV differs from the oracle (state {sf[i][:3]}, path {si[i][:10]})"
        on_node = bool((env.map.lp_nodes == sf[i, :2]).all(1).any())
        counts += (1, r, r * on_node)
    return counts


def report(what, counts):
    """prints the counts and fails when more than 0.1 % of the frames of cars off the lanepath nodes needed the one-ulp cos/sin
    nudge: away from the degenerate poses check_frames describes, a last-bit difference of cos/sin almost never moves a pixel, so
    frequent nudges would mean the device's cos/sin are further off"""
    frames, nudged, on_node = (int(v) for v in counts)
    print(f"{what}: {frames} BEV frames equal to the oracle, {nudged} of them with cos/sin moved by one ulp "
          f"({on_node} with the car on a lanepath node)")
    assert (nudged - on_node) * 1000 <= frames, f"{what}: {nudged - on_node} of {frames} frames off the lanepath nodes needed the nudge"


@pytest.mark.parametrize("map_name", ["knuffingen", "simple_layout"])
def test_bev_rollout_matches_oracle(map_name):
    n, steps = 2048, 30
    env = TinyCarloVecEnv(bev_config(map_name, bev=BEV), n, device="cuda:0", autoreset="next_step")
    rng = np.random.default_rng(7)
    env.reset(seed=3)
    counts = check_frames(env)
    drawn = 0
    for t in range(steps):
        _, _, _, _, info = env.step(actions(rng, n, t, env.device))
        assert info["bev"] is env.bev
        counts += check_frames(env)
        drawn += int(env.bev.flatten(1).any(1).sum().item())
    report(map_name, counts)
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
    report("headline size (sampled)", check_frames(env, envs=ids))


# ------------------------------------------------------------------------------------------------ geometry table
def shaped_config(map_name, tmp_path, bev, cam=None):
    """a config on a bundled map or on one of map_shapes_util's regrouped Knuffingen maps, with a `bev` section"""
    cfg = make_config("knuffingen" if map_name in M.MAPS else map_name, "classes", cam=cam)
    if map_name in M.MAPS:
        cfg["map"] = {"json_path": M.write(M.MAPS[map_name](), tmp_path, map_name), "pixel_per_meter": M.PPM,
                      "spawn_points": list(M.SPAWN_KNUFF)}
    cfg["bev"] = dict(bev)
    return cfg


def poison(env):
    env.bev.view(torch.uint8).fill_(0xAB)


def poisoned(env):
    """bool [N]: the envs whose whole BEV still holds the poison"""
    return (env.bev.view(torch.uint8).flatten(1) == 0xAB).all(1).cpu().numpy()


# id: (map, `bev` section, envs). Knuffingen and simple_layout have 5 classes, the formula student maps 3.
GEOMETRY = {
    **{f"t{t}": ("knuffingen", dict(BEV, line_thickness=t), 48) for t in (1, 3, 4, 5, 6, 7, 8)},
    # planes that start part-way into a word, env bases that are not 16-byte aligned (npx = P*H*W bytes per env)
    "75x100": ("knuffingen", dict(BEV, resolution=[75, 100], line_thickness=3), 48),
    "33x35": ("knuffingen", dict(BEV, resolution=[33, 35], pixel_per_meter=60), 48),
    "129x129": ("simple_layout", dict(BEV, resolution=[129, 129], line_thickness=4), 48),
    "1x1": ("knuffingen", dict(BEV, resolution=[1, 1], car_pixel=[0.5, 0.5], line_thickness=3), 48),   # npx = 6
    # extreme aspect ratios
    "1x4096": ("knuffingen", dict(BEV, resolution=[1, 4096]), 32),
    "4096x1": ("knuffingen", dict(BEV, resolution=[4096, 1], line_thickness=5), 32),
    "7x1001": ("knuffingen", dict(BEV, resolution=[7, 1001], line_thickness=5, pixel_per_meter=200), 32),
    # plane count: 1, 2, 3 and 16 planes; K16 has a zero-length edge (a disc), a class of nodes only and an empty class
    "K1": ("K1", dict(BEV, route=False), 48),
    "K1_route": ("K1", dict(BEV, line_thickness=3), 48),
    "K2_route": ("K2", dict(BEV, resolution=[96, 96], line_thickness=1), 48),
    "K15_route": ("K15", dict(BEV, resolution=[96, 96], pixel_per_meter=100), 48),
    "K16R": ("K16R", dict(BEV, resolution=[96, 96], route=False, line_thickness=3), 48),
    "K16": ("K16", dict(BEV, route=False, pixel_per_meter=200), 48),
    # scale: the whole map in a few pixels (heavy overdraw) up to endpoints beyond int32 (INT_MIN by the contract)
    "ppm2": ("knuffingen", dict(BEV, pixel_per_meter=2, line_thickness=3), 48),
    "ppm25": ("knuffingen", dict(BEV, pixel_per_meter=25), 48),
    "ppm1000": ("knuffingen", dict(BEV, pixel_per_meter=1000, line_thickness=4), 48),
    "ppm1e6": ("knuffingen", dict(BEV, pixel_per_meter=1e6), 48),
    "ppm1e9": ("knuffingen", dict(BEV, pixel_per_meter=1e9, line_thickness=8), 48),
    # car pixel
    "car_centre": ("knuffingen", dict(BEV, resolution=[96, 128], car_pixel=[64.0, 48.0]), 48),
    "car_bottom_row": ("knuffingen", dict(BEV, resolution=[96, 128], car_pixel=[63.5, 95.0], line_thickness=3), 48),
    "car_fractional_negative": ("knuffingen", dict(BEV, resolution=[96, 128], car_pixel=[-3.75, -0.5]), 48),
    "car_far_outside": ("knuffingen", dict(BEV, resolution=[96, 128], car_pixel=[-150.0, 600.0], pixel_per_meter=300), 48),
    # bit-packed, against pack_bits(oracle); 96x100: W is not a multiple of 32
    "bits_96x100": ("knuffingen", dict(BEV, resolution=[96, 100], format="classes_bits", line_thickness=3), 48),
    "bits_8x4": ("knuffingen", dict(BEV, resolution=[8, 4], format="classes_bits", pixel_per_meter=20), 48),
    "bits_128x128": ("knuffingen", dict(BEV, format="classes_bits"), 48),
    # the four bundled maps at other geometries
    "map_knuffingen": ("knuffingen", dict(BEV, resolution=[100, 150], pixel_per_meter=90, line_thickness=3, route=False), 48),
    "map_simple_layout": ("simple_layout", dict(BEV, resolution=[64, 200], pixel_per_meter=150, line_thickness=1, car_pixel=[100.0, 32.0]), 48),
    "map_formula_student_track": ("formula_student_track", dict(BEV, resolution=[120, 90], pixel_per_meter=20), 32),
    "map_formula_student_skidpad": ("formula_student_skidpad", dict(BEV, resolution=[80, 80], pixel_per_meter=15, line_thickness=4,
                                                                    format="classes_bits"), 32),
    # the largest frames the stacked plane accepts (test_bev_shared_memory_bound): 204 688 and 204 784 of 204 800 bytes
    "smem_6x512x533": ("knuffingen", dict(BEV, resolution=[512, 533], pixel_per_meter=64, line_thickness=3), 24),
    "smem_16x316x324": ("K15", dict(BEV, resolution=[316, 324], pixel_per_meter=100), 24),
    # env counts: one block, and a grid that is not a multiple of anything
    "n1": ("knuffingen", dict(BEV, resolution=[33, 35], line_thickness=3), 1),
    "n4099": ("knuffingen", dict(BEV, resolution=[33, 35], line_thickness=3), 4099),
}


@pytest.mark.parametrize("case", list(GEOMETRY))
def test_bev_geometry_matches_oracle(case, tmp_path):
    """reset, 8 steps with next-step autoresets (a quarter of the envs marked done at step 3), a masked reset: every env's BEV on
    every step equals the oracle; the masked reset leaves the deselected envs' BEV alone"""
    map_name, bev, n = GEOMETRY[case]
    seed = list(GEOMETRY).index(case)
    env = TinyCarloVecEnv(shaped_config(map_name, tmp_path, bev, cam={"resolution": [64, 64]}), n, device="cuda:0", autoreset="next_step")
    assert env.bev_cfg["planes"] == env.n_classes + int(bev["route"])
    rng = np.random.default_rng(seed)
    poison(env)
    env.reset(seed=seed)
    counts = check_frames(env)
    drawn = int(env.bev.flatten(1).any(1).sum().item())
    autoresets = 0
    for t in range(8):
        if t == 3:
            env.mark_done(torch.from_numpy(np.arange(n) % 4 == 0).to(env.device))
        poison(env)
        env.step(actions(rng, n, t, env.device))
        autoresets += int(env.reset_mask.sum().item())
        counts += check_frames(env)
        drawn += int(env.bev.flatten(1).any(1).sum().item())
    mask = rng.random(n) < 0.5
    mask[0] = True
    poison(env)
    env.reset(mask=torch.from_numpy(mask))
    assert poisoned(env)[~mask].all() and not poisoned(env)[mask].any()
    counts += check_frames(env, envs=np.nonzero(mask)[0])
    report(f"{case} ({env.bev_cfg['planes']} planes, {drawn} frames drew)", counts)
    assert autoresets >= (n + 3) // 4
    assert drawn > 0


@pytest.mark.parametrize("map_name,classes,ok,bad", [("knuffingen", 5, (512, 533), (512, 534)), ("K15", 15, (316, 324), (316, 325))])
def test_bev_shared_memory_bound(map_name, classes, ok, bad, tmp_path):
    """the largest stacked plane (P*H*W bits + a pad word, in 16-byte units) that fits 200 KB is accepted, one column more is
    rejected, by bev_params and by tc_set_bev called through the ABI"""
    def smem(H, W):
        return ((((classes + 1) * H * W + 31) // 32 + 1) * 4 + 15) // 16 * 16
    assert smem(*ok) <= BEV_SMEM_MAX < smem(*bad)
    cfg = shaped_config(map_name, tmp_path, {"resolution": list(ok), "route": True})
    assert bev_params(cfg, classes)["planes"] == classes + 1
    with pytest.raises(ValueError, match="shared memory"):
        bev_params(dict(cfg, bev={"resolution": list(bad), "route": True}), classes)
    env = TinyCarloVecEnv(cfg, 3, device="cuda:0")
    L = env._L
    for fmt in (_lib.TC_OBS_CLASSES, _lib.TC_OBS_CLASSES_BITS):
        d = _lib.TcBevDesc(bad[0], bad[1], 128.0, bad[1] / 2, bad[0] * 7 / 8, 1, 1, fmt)
        assert L.tc_set_bev(env._h, C.byref(d), C.c_void_p(env.bev.data_ptr())) != 0
        # 316x325 is not bit-packable either: for that format the first rule that fails may be the word rule
        assert b"shared memory" in L.tc_last_error() or (fmt == _lib.TC_OBS_CLASSES_BITS and bad[0] * bad[1] % 32)
    # accepted in u8, and bit-packed where H*W is a multiple of 32 (512x533; 316x324 is not); the handle then renders it
    packable = ok[0] * ok[1] % 32 == 0
    bev = {"resolution": list(ok), "route": True, "format": "classes_bits" if packable else "classes"}
    env.bev_cfg = bev_params(dict(cfg, bev=bev), classes)
    env.bev = (torch.zeros((3, classes + 1, ok[0] * ok[1] // 32), dtype=torch.int32, device=env.device) if packable else
               torch.zeros((3, classes + 1) + ok, dtype=torch.uint8, device=env.device))
    fmt = _lib.TC_OBS_CLASSES_BITS if packable else _lib.TC_OBS_CLASSES
    d = _lib.TcBevDesc(ok[0], ok[1], env.bev_cfg["pixel_per_meter"], *env.bev_cfg["car_pixel"], 1, 1, fmt)
    assert L.tc_set_bev(env._h, C.byref(d), C.c_void_p(env.bev.data_ptr())) == 0
    env.reset(seed=1)
    report(f"{map_name} at {ok[0]}x{ok[1]} {bev['format']}", check_frames(env))
    assert env.bev.any()


# ------------------------------------------------------------------------------------------------ placed poses
def parallel_poses(tables, H, W, k, col0, row0, t):
    """states [n,8] that put Knuffingen's longest laneline edge (0.58 m) parallel to each side of the frame, centred on it and
    d = 0, t/2, (t+1)/2, t+1, t+2 pixels outside it (on the frame's outer row / column for d = 0), at headings up to 3 turns
    beyond +-pi. tc_bev_segment culls a segment whose endpoints both lie more than t+1 pixels beyond one side."""
    best = None
    for c in range(tables.n_classes):
        nodes, edges = tables.class_nodes(c), tables.class_edges(c)
        L = np.hypot(*(nodes[edges[:, 1]] - nodes[edges[:, 0]]).T)
        j = int(L.argmax())
        if best is None or L[j] > best[0]:
            best = (L[j], nodes[edges[j, 0]], nodes[edges[j, 1]])
    L, a, b = best
    assert L * k > max(H, W)   # the edge crosses the whole frame
    e, mid = (b - a) / L, (a + b) / 2
    rows = []
    for side in ("top", "bottom", "left", "right"):
        for d in sorted({0, t // 2, (t + 1) // 2, t + 1, t + 2}):
            target = {"top": -d, "bottom": H - 1 + d, "left": -d, "right": W - 1 + d}[side]
            at = target + (0.5 if target >= 0 else -0.5)   # mid-pixel: truncation lands on `target`
            if side in ("top", "bottom"):     # the edge horizontal in the image
                c, s, u, v = e[1], -e[0], W / 2, at
            else:                             # vertical
                c, s, u, v = e[0], e[1], at, H / 2
            f, r = np.array([c, s]), np.array([-s, c])
            car = mid - (u - col0) / k * r - (row0 - v) / k * f
            for turns in (0, -3, 2):
                rows.append([car[0], car[1], math.atan2(s, c) + 2 * math.pi * turns])
    return np.array(rows)


@pytest.mark.parametrize("t", range(1, 9))
def test_bev_placed_poses_at_the_culling_margin(t):
    """load_state_dict + render_bev at poses that put a long laneline edge just inside, on and beyond the culling margin of
    each frame side; cars with path_len 0..4 (the route plane); cars whose state is NaN (every endpoint INT_MIN)"""
    H, W, k = 48, 64, 200.0
    bev = {"resolution": [H, W], "pixel_per_meter": k, "line_thickness": t, "route": True}
    cfg = bev_config("knuffingen", bev=bev, cam={"resolution": [64, 64]})
    tables = MapTables(f"{MAPS_DIR}/knuffingen.json", PPM["knuffingen"])
    col0, row0 = W / 2, 7 * H / 8
    place = parallel_poses(tables, H, W, k, col0, row0, t)
    rng = np.random.default_rng(t)
    n_route, n_nan = 10, 2
    n = len(place) + n_route + n_nan
    sf = np.zeros((n, 8))
    si = np.full((n, 16), -1, np.int32)
    si[:, 0] = 0
    sf[:len(place), :3] = place
    for i in range(len(place), len(place) + n_route):   # on a lanepath node, path_len = 0..4 consecutive edges
        sf[i, :2] = tables.lp_nodes[rng.integers(len(tables.lp_nodes))] + rng.normal(0, 0.05, 2)
        sf[i, 2] = rng.uniform(-3 * math.pi, 3 * math.pi)
        si[i, 0] = (i - len(place)) % 5
        for j in range(si[i, 0]):
            si[i, 2 + 2 * j:4 + 2 * j] = tables.lp_edges[rng.integers(len(tables.lp_edges))]
    sf[n - n_nan:, :3] = np.nan
    si[n - n_nan:, 0] = 4
    si[n - n_nan:, 2:10] = tables.lp_edges[:4].reshape(-1)
    env = TinyCarloVecEnv(cfg, n, device="cuda:0")
    env.reset(seed=0)
    env.load_state_dict({"sf": torch.from_numpy(sf), "si": torch.from_numpy(si)})
    poison(env)
    env.render_bev()
    report(f"thickness {t}, placed poses", check_frames(env))
    b = env.bev.cpu().numpy()
    assert not b[n - n_nan:].any()
    # the edge on the frame's outer row / column is drawn; a thick one reaches in from outside too
    per = len(place) // 4
    inside = [b[s * per:(s + 1) * per].any() for s in range(4)]
    assert all(inside), inside


# ------------------------------------------------------------------------------------------------ memory safety, entry points
@pytest.mark.parametrize("fmt,res", [("classes", (75, 100)), ("classes_bits", (96, 100)), ("classes", (512, 533)), ("classes_bits", (512, 533))])
def test_bev_guard_bands_determinism_and_full_overwrite(fmt, res):
    """tc_set_bev pointed at a payload inside [guard | payload | guard] (u8 payload 3 bytes past a 16-byte boundary, bits one word
    past it; 75x100 is not bit-packable, hence 96x100): the sentinels survive, the payload poisoned with 0xAB before every step
    comes back equal to the oracle, and the same step from the same state six times over gives bit-identical frames (the planes
    are drawn with shared-memory atomicOr: a missing barrier would make them depend on timing)"""
    H, W = res
    n = 7 if H > 100 else 21
    bev = {"resolution": [H, W], "pixel_per_meter": 90.0, "line_thickness": 3, "route": True, "format": fmt}
    env = TinyCarloVecEnv(bev_config("knuffingen", bev=bev, cam={"resolution": [64, 64]}), n, device="cuda:0")
    G, off = 4096, 3 if fmt == "classes" else 4
    nb = env.bev.numel() * env.bev.element_size()
    buf = torch.full((G + off + nb + G,), 0x5C, dtype=torch.uint8, device=env.device)
    env.bev = buf[G + off:G + off + nb].view(env.bev.dtype).view(env.bev.shape)
    b = env.bev_cfg
    d = _lib.TcBevDesc(H, W, b["pixel_per_meter"], b["car_pixel"][0], b["car_pixel"][1], b["line_thickness"], 1,
                       _lib.TC_OBS_CLASSES_BITS if fmt == "classes_bits" else _lib.TC_OBS_CLASSES)
    _lib.check(env._L.tc_set_bev(env._h, C.byref(d), C.c_void_p(env.bev.data_ptr())), "tc_set_bev")

    def guards_intact():
        g = buf.cpu().numpy()
        return (g[:G + off] == 0x5C).all() and (g[G + off + nb:] == 0x5C).all()
    rng = np.random.default_rng(17)
    poison(env)
    env.reset(seed=6)
    counts = check_frames(env)
    for t in range(3):
        a = actions(rng, n, t, env.device)
        st0 = {k: v.clone() for k, v in env.state_dict().items()}
        first = None
        for rep in range(6):
            env.load_state_dict(st0)
            poison(env)
            env.step(a)
            if first is None:
                first = env.bev.clone()
                counts += check_frames(env)
            else:
                assert torch.equal(env.bev, first), f"step {t}, repetition {rep}: the BEV differs"
        assert guards_intact(), f"step {t}: a guard band was overwritten"
    assert first.any()
    report(f"{fmt} {H}x{W} in guard bands", counts)


def test_bev_step_f64_step_host_and_restore():
    """the BEV after tc_step_f64 (float64 actions), tc_step_host and restore (tc_set_state + tc_render_bev) equals the oracle"""
    n = 64
    bev = {"resolution": [75, 100], "pixel_per_meter": 100, "line_thickness": 3, "route": True}
    env = TinyCarloVecEnv(bev_config("knuffingen", bev=bev, cam={"resolution": [64, 64]}), n, device="cuda:0", autoreset="next_step")
    rng = np.random.default_rng(12)
    env.reset(seed=12)
    counts = check_frames(env)
    for t in range(3):
        a = actions(rng, n, t, env.device)
        a["car_control"] = a["car_control"].double()
        poison(env)
        env.step(a)
        counts += check_frames(env)
    reward, term, trunc = torch.zeros(n), torch.zeros(n, dtype=torch.uint8), torch.zeros(n, dtype=torch.uint8)
    for t in range(3):
        a = actions(rng, n, t, env.device)
        poison(env)
        env.step_host(a["car_control"].cpu(), a["maneuver"].cpu(), reward, term, trunc)
        counts += check_frames(env)
    ck = env.checkpoint()
    want = env.bev.clone()
    env.step(actions(rng, n, 0, env.device))
    assert not torch.equal(env.bev, want)
    poison(env)
    env.restore(ck)
    assert torch.equal(env.bev, want)
    counts += check_frames(env)
    report("tc_step_f64, tc_step_host, restore", counts)


def test_bev_on_a_rig_is_per_env():
    """a camera rig (M = 3) gives the BEV of the one-camera env, env for env; its masked tc_reset and tc_render_bev select envs,
    not views: deselected envs keep the poison, selected ones equal the oracle, and a selected env whose reset fails (spawn
    node -1) is rendered at its old pose"""
    n = 64
    bev = {"resolution": [75, 100], "pixel_per_meter": 100, "line_thickness": 2, "route": True}
    plain = bev_config("knuffingen", bev=bev, cam={"resolution": [64, 64]})
    rig = dict(plain, cameras=[{}, REAR, {"fov": 110}])
    envs = [TinyCarloVecEnv(c, n, device="cuda:0", autoreset="next_step") for c in (rig, plain)]
    assert envs[0].n_cameras == 3
    rng = np.random.default_rng(3)
    for e in envs:
        e.reset(seed=3)
    assert torch.equal(envs[0].bev, envs[1].bev)
    for t in range(4):
        a = actions(rng, n, t, envs[0].device)
        for e in envs:
            e.step(a)
        assert torch.equal(envs[0].bev, envs[1].bev), f"step {t}"
    env = envs[0]
    mask = rng.random(n) < 0.5
    mask[:4] = [True, False, True, False]
    nodes = env._spawn_nodes.cpu().numpy().copy()
    nodes[2] = -1   # env 2's reset fails
    old = env.state_dict()["sf"].cpu().numpy()
    poison(env)
    env.reset(mask=torch.from_numpy(mask), spawn_nodes=torch.from_numpy(nodes))
    assert np.array_equal(env.state_dict()["sf"].cpu().numpy()[2], old[2])
    assert poisoned(env)[~mask].all() and not poisoned(env)[mask].any()
    counts = check_frames(env, envs=np.nonzero(mask)[0])
    poison(env)
    env.render_bev(mask=torch.from_numpy(~mask))
    assert poisoned(env)[mask].all() and not poisoned(env)[~mask].any()
    counts += check_frames(env, envs=np.nonzero(~mask)[0])
    report("rig, masked reset and render", counts)
