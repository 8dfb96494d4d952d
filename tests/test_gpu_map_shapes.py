"""GPU parity on maps with 1, 2 and 16 laneline classes and per-env line thicknesses from 1 to 255, through every render path.

The bundled maps have 3 or 5 classes and the other device tests draw lines 1 to 6 pixels thick, yet much of the render code
depends on the class count (which kernel a frame size takes, band counts, class fields packed into bytes, painter's order of
the RGB composition, per-class tracking outputs) and on the thickness (bands and primitive lists of the banded kernels). The
maps are Knuffingen regrouped (tests/map_shapes_util.py): K1, K2, K16 (edges dealt one by one over 13 classes, plus a class
with nodes only, an empty class and a zero-length edge) and K16R (the same, dealt in runs of 16 edges, which keeps the union
graph small enough for the small-frame block-per-env kernels).

Every case asserts the render path it covers, from render_info() and the kernel launches per step, so that a change of
tc_render_path cannot quietly move it to another kernel. Where tc_render_path's rule differs from what one might expect
for a frame size, the case follows the rule and says so:
  * K16 never takes the block-per-env small-frame kernels: single-edge dealing puts almost every node into two classes, and
    the whole-graph tables of that union exceed the 100 KB of tc_create's fused_all rule. K16R covers those kernels instead;
  * K16R at 128x160 takes the one-env kernel by the rule (two 16-plane envs per block do not fit 3 blocks per SM); the
    packed kernel is covered at 64x96;
  * K16 bit-packed at 128x160 takes the two-kernel primitives path; K1 at 480x640 fits one block per env (one plane).
Each step every env is compared with the CPU oracle: frames bit for bit (the buffer is poisoned with 0xAB first, so a
skipped store shows), info_f64 to 1e-9 relative, nearest_edge, terminated and truncated exactly."""
import os
import zlib

import numpy as np
import pytest
import torch

import map_shapes_util as M
from oracle import oracle as orc
from pair_util import make_config
from test_gpu_parity import _check_segments

pytestmark = pytest.mark.gpu

RTOL64 = 1e-9
LAUNCHES = {"packed": 2, "one_env": 2, "per_class": 2, "banded": 2, "prims": 4, "unfused": 3}   # tracking + render per step

# id: (map, obs format, resolution, envs, camera overrides, environment at construction, path tc_render_path takes)
CASES = {
    "K1_classes_84x84": ("K1", "classes", [84, 84], 128, {}, {}, "packed"),
    "K2_classes_128x160": ("K2", "classes", [128, 160], 128, {}, {}, "packed"),
    "K16R_classes_64x96": ("K16R", "classes", [64, 96], 96, {}, {}, "packed"),
    "K16R_bits_64x96": ("K16R", "classes_bits", [64, 96], 96, {}, {}, "packed"),
    "K16R_bf16_64x96": ("K16R", "classes_bf16", [64, 96], 96, {}, {}, "packed"),
    "K16R_rgb_64x96": ("K16R", "rgb", [64, 96], 96, {}, {}, "packed"),
    "K16R_classes_128x160": ("K16R", "classes", [128, 160], 64, {}, {}, "one_env"),
    "K16R_classes_84x84_pack0": ("K16R", "classes", [84, 84], 64, {}, {"TC_ENV_PACK": "0"}, "one_env"),
    "K16_classes_128x160": ("K16", "classes", [128, 160], 64, {}, {}, "per_class"),
    "K16_bf16_128x160": ("K16", "classes_bf16", [128, 160], 64, {}, {}, "per_class"),
    "K16_bits_128x160": ("K16", "classes_bits", [128, 160], 64, {}, {}, "prims"),
    "K16_rgb_96x128": ("K16", "rgb", [96, 128], 64, {}, {}, "banded"),
    "K16_classes_240x320": ("K16", "classes", [240, 320], 32, {}, {}, "per_class"),
    "K1_classes_480x640": ("K1", "classes", [480, 640], 16, {}, {}, "one_env"),
    "K16_classes_480x640": ("K16", "classes", [480, 640], 16, {}, {}, "per_class"),
    "K16_bf16_480x640": ("K16", "classes_bf16", [480, 640], 16, {}, {}, "per_class"),
    "K16_bits_480x640_far": ("K16", "classes_bits", [480, 640], 16, {"max_range": 3.0, "orientation": [30, 0, 0]}, {}, "prims"),
    "K16_rgb_480x640": ("K16", "rgb", [480, 640], 16, {}, {}, "banded"),
    "K16_rgb_544x640": ("K16", "rgb", [544, 640], 16, {}, {}, "banded"),
    "K16_classes_128x160_segments": ("K16", "classes", [128, 160], 64, {}, {}, "unfused"),
}


def render_path(env):
    """the render path env's steps take, read from render_info() with the conditions of tc_render_path (tc_api.cu)"""
    ri = env.render_info()
    fmt = env.observation_space_format
    if "seg_count" in env.out:
        return "unfused"
    if ri["block_per_env"]:
        return "packed" if ri["envs_per_block"] > 0 else "one_env"
    px = env.H * env.W
    if ri["banded_smem"] > 0 and fmt == "classes_bits" and px % 128 == 0 and ((px + 31) // 32 + 1) * 4 <= 64 * 1024:
        return "prims"
    if ri["banded_smem"] > 0 and fmt in ("classes_bits", "rgb"):
        return "banded"
    if ri["render_smem"] <= 56 * 1024 and fmt != "rgb":
        return "per_class"
    return "unfused"


def banded_bands(H, W, C):
    """band count of tc_render_env_banded_kernel: tc_band_geometry(H, W, C + 1 planes, 30 KB) in tc_api.cu"""
    planes, budget = C + 1, 30 * 1024
    words = lambda r: (r * W + 31) // 32 + 1   # noqa: E731
    rows = H
    while rows > 1 and words(rows) * 4 * planes > budget:
        rows = (rows + 1) // 2
    if rows < H:
        rows = (rows + 15) // 16 * 16
        while rows > 16 and words(rows) * 4 * planes > budget:
            rows -= 16
        rows = min(rows, H)
    return (H + rows - 1) // rows


def decode(obs, fmt, H, W):
    """the observation as the oracle's u8 masks / RGB frames"""
    if fmt == "classes_bf16":
        f = obs.float().cpu().numpy()
        assert set(np.unique(f)).issubset({0.0, 1.0}), "bf16 masks must hold 0.0 / 1.0 only"
        return (f * 255).astype(np.uint8)
    o = obs.cpu().numpy()
    if fmt == "classes_bits":
        n = o.shape[0]
        return np.unpackbits(o.view(np.uint32).view(np.uint8), axis=-1, bitorder="little")[..., : H * W].reshape(n, -1, H, W) * 255
    return o


def _build(case, tmp_path):
    map_name, fmt, res, n, cam, setenv, _ = CASES[case]
    data = M.MAPS[map_name]()
    cfg = make_config("knuffingen", "rgb" if fmt == "rgb" else "classes", cam=dict(resolution=res, **cam))
    cfg["map"] = {"json_path": M.write(data, tmp_path, map_name), "pixel_per_meter": M.PPM, "spawn_points": list(M.SPAWN_KNUFF)}
    th = np.resize(np.array(M.THICKNESSES, np.int32), n)
    from tinycarlo_b200 import TinyCarloVecEnv
    old = {k: os.environ.get(k) for k in setenv}
    os.environ.update(setenv)
    try:   # the visible-set tables (and with them the packed kernel's geometry) are rebuilt by set_camera_params
        env = TinyCarloVecEnv(cfg, n, device="cuda:0", obs_format=None if fmt in ("classes", "rgb") else fmt,
                              debug_segments=case.endswith("_segments"))
        env.set_camera_params(line_thickness=th)
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
    assert np.array_equal(env._thickness, th)
    omap = orc.OracleMap(data, M.PPM, M.SPAWN_KNUFF)
    oenv = orc.OracleVecEnv(omap, n, env._car_rows.copy(), env._cam_rows.copy(), th, res[0], res[1], "rgb" if fmt == "rgb" else "classes")
    return env, oenv, fmt, res


def _compare(env, oenv, fmt, H, W, where):
    got = decode(env.obs, fmt, H, W)
    bad = np.nonzero((got != oenv.obs).reshape(got.shape[0], -1).any(axis=1))[0]
    if len(bad):
        i = int(bad[0])
        diff = np.argwhere(got[i] != oenv.obs[i])
        pytest.fail(f"{where}: {len(bad)} of {got.shape[0]} frames differ from the oracle; env {i} (thickness {int(oenv.thick[i])}): "
                    f"{len(diff)} values, first at {diff[:3].tolist()}")
    return got.shape[0]


def _compare_info(env, oenv, where):
    np.testing.assert_allclose(env.out["info_f64"].cpu().numpy(), oenv.info, rtol=RTOL64, atol=1e-11, err_msg=f"info {where}")
    assert np.array_equal(env.out["nearest_edge"].cpu().numpy(), oenv.nearest), f"nearest laneline edge {where}"
    assert np.array_equal(env.out["terminated"].cpu().numpy(), oenv.terminated), f"terminated {where}"
    assert np.array_equal(env.out["truncated"].cpu().numpy(), oenv.truncated), f"truncated {where}"


@pytest.mark.parametrize("case", list(CASES))
def test_cuda_map_shapes_match_oracle(case, tmp_path):
    map_name, fmt, res, n, cam, setenv, want_path = CASES[case]
    H, W = res
    env, oenv, fmt, res = _build(case, tmp_path)
    path = render_path(env)
    assert path == want_path, (case, path, env.render_info())
    if case.startswith("K16_rgb_") and H >= 480:
        assert banded_bands(H, W, env.n_classes) == {480: 30, 544: 34}[H]   # 544 rows: more than 32 bands, the all-bands mask
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    stats = {"frames": 0, "steps": 0, "resets": 0, "most_segments": 0}
    spawn = rng.choice(M.SPAWN_KNUFF, n).astype(np.int32)
    spawn[0] = M.SPAWN_KNUFF[0]   # env 0 starts behind K16's zero-length edge
    env.obs.view(torch.uint8).fill_(0xAB)
    env.reset(seed=zlib.crc32(case.encode()) & 0xFFFF, spawn_nodes=torch.from_numpy(spawn))
    oenv.reset(spawn)
    stats["frames"] += _compare(env, oenv, fmt, H, W, "reset")
    if map_name.startswith("K16") and fmt != "rgb":   # the zero-length edge is seen (a disc, or one pixel at thickness 1)
        assert oenv.obs[0, M.K16_DOT].any(), "env 0 does not see the zero-length edge"
        assert not oenv.obs[:, [M.K16_EMPTY, M.K16_NODES_ONLY]].any()
    seg_stats = {"near": 0, "far": 0, "far_diff": 0}
    for t in range(8):
        cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
        man = rng.integers(0, 4, n).astype(np.int32)
        env.obs.view(torch.uint8).fill_(0xAB)
        l0 = env.launch_count
        env.step({"car_control": torch.from_numpy(cc).cuda(), "maneuver": torch.from_numpy(man).cuda()})
        assert env.launch_count - l0 == LAUNCHES[want_path], (case, env.launch_count - l0)
        oenv.step(cc.astype(np.float64), man)
        stats["frames"] += _compare(env, oenv, fmt, H, W, f"step {t}")
        stats["steps"] += 1
        _compare_info(env, oenv, f"step {t}")
        if map_name.startswith("K16"):   # classes without edges: distance 0, no nearest edge, on both sides
            got_d, got_e = env.out["info_f64"][:, 4:].cpu().numpy(), env.out["nearest_edge"].cpu().numpy()
            for c in (M.K16_EMPTY, M.K16_NODES_ONLY):
                assert (oenv.dist[:, c] == 0).all() and (oenv.nearest[:, c] == -1).all(), c
                assert (got_d[:, c] == 0).all() and (got_e[:, c] == -1).all(), c
        if want_path in ("prims", "unfused"):
            counts = [oenv.segments(i) for i in range(n)]
            stats["most_segments"] = max(stats["most_segments"], max(int(c[0].sum()) for c in counts))
        if want_path == "unfused":
            off = env.map.ll_edge_off
            cnt = env.out["seg_count"].cpu().numpy()
            seg = env.out["seg_i32"].cpu().numpy()
            for i, (ocnt, oseg, _, _) in enumerate(counts):
                assert np.array_equal(cnt[i], ocnt), (t, i)
                for c in range(env.n_classes):
                    _check_segments(seg[i, off[c]:off[c] + cnt[i, c]], oseg[off[c]:off[c] + ocnt[c]], (case, t, i, c), seg_stats)
        done = (oenv.terminated | oenv.truncated).astype(bool)
        if done.any():
            env.reset_done()
            oenv.reset(env._spawn_nodes.cpu().numpy(), mask=done)
            _compare(env, oenv, fmt, H, W, f"reset after step {t}")
            stats["frames"] += int(done.sum())
            stats["resets"] += int(done.sum())
    if case == "K16_bits_480x640_far":   # envs beyond the 64 segments of the primitive lists go to the banded kernel
        assert stats["most_segments"] > 64, stats
    assert oenv.obs.any()
    print(f"{case}: path {path}, {stats}, segments {seg_stats}")
    env.close()
