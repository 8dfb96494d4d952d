"""GPU tests of the blob-noise kernel (tc_noise_blobs / NoiseObservationWrapper) against the reference's operation
(tests/noise_util.py: tinycarlo/wrapper/observation.py:14-27 with cv2, driven by the header's Philox draws).

The kernel is called through the ABI of a real handle on a caller-owned buffer of random bytes (so that every OR and every
erase shows) between sentinel guard bands, over the geometry table of noise_util.GEOMETRY: 1, 2, 3, 5 and 16 classes, frames
from 1x1 to 480x640, radii 1 to 1023, 0 to 37 blobs, extreme seeds and steps, offsets across 2^31, masks and rigs, plus a
buffer larger than 2^31 bytes. Then the wrapper: a 480x640 rollout with autoresets, the single-env drop-in, the formats it
leaves alone, and the grouped env, whole and sharded."""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")

import map_shapes_util as MS  # noqa: E402
from noise_util import CLASSES, GEOMETRY, M32, expected_noise, geometry_id, make_mask, reference_noise  # noqa: E402
from pair_util import make_config  # noqa: E402
from rig_util import REAR  # noqa: E402

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
GUARD = 4096            # sentinel bytes on each side of the buffer
TC_ERR_INVALID = -1
RIG = [{}, REAR, {"fov": 110}]


@pytest.fixture(scope="module")
def map_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("noise_maps")


def config(mp, H, W, M, map_dir, fmt="classes"):
    if mp in MS.MAPS:
        cfg = make_config("knuffingen", fmt, cam={"resolution": [H, W]})
        cfg["map"] = {"json_path": MS.write(MS.MAPS[mp](), map_dir, mp), "pixel_per_meter": MS.PPM, "spawn_points": list(MS.SPAWN_KNUFF)}
    else:
        cfg = make_config(mp, fmt, cam={"resolution": [H, W]})
    if M > 1:
        cfg["cameras"] = RIG[:M]
    return cfg


def handle(mp, N, M, H, W, map_dir):
    from tinycarlo_b200 import TinyCarloVecEnv
    env = TinyCarloVecEnv(config(mp, H, W, M, map_dir), N, device=DEV)
    assert (env.num_envs, env.n_cameras, env.H, env.W) == (N, M, H, W) and len(env.class_names) == CLASSES[mp]
    return env


def noise(env, buf, seed, step, n_blobs, max_radius, offset, mask=None):
    """tc_noise_blobs on the views that start GUARD bytes into buf (u8, on the device); returns the library's return code"""
    torch.cuda.synchronize()
    return env._L.tc_noise_blobs(env._h, C.c_void_p(buf.data_ptr() + GUARD), int(seed) & (2**64 - 1), int(step) & M32, int(n_blobs),
                                 int(max_radius), int(offset), None if mask is None else C.c_void_p(mask.data_ptr()),
                                 C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream))


def guarded(shape, rng):
    """(device buffer with guard bands, its host copy, the views [N, M, C, H, W] of the host copy)"""
    n = int(np.prod(shape))
    host = rng.integers(0, 256, n + 2 * GUARD, dtype=np.uint8)
    return torch.from_numpy(host).to(DEV), host, host[GUARD:GUARD + n].reshape(shape)


def check_call(env, row, mask, buf, before, sample=None):
    """one call on buf (holding `before`, a host copy): rc, guard bands, the sampled envs' views against the reference,
    the unselected envs' views unchanged, and a second call on the same input bit-identical to the first"""
    mp, N, M, H, W, r, nb, seed, step, off, _ = row
    n = N * M * CLASSES[mp] * H * W
    mask_d = None if mask is None else torch.from_numpy(mask).to(DEV)
    assert noise(env, buf, seed, step, nb, r, off, mask_d) == 0
    first = buf.clone()
    got = first.cpu().numpy()
    assert np.array_equal(got[:GUARD], before[:GUARD]) and np.array_equal(got[GUARD + n:], before[GUARD + n:]), "guard band written"
    shape = (N, M, CLASSES[mp], H, W)
    views, was = got[GUARD:GUARD + n].reshape(shape), before[GUARD:GUARD + n].reshape(shape)
    envs = range(N) if sample is None else sample
    want = expected_noise(was, row, mask, envs)
    for i in envs:
        assert np.array_equal(views[i], want[i]), ("env", i)
    if mask is not None:
        assert np.array_equal(views[mask == 0], was[mask == 0]), "an unselected env's views changed"
    buf.copy_(torch.from_numpy(before))
    assert noise(env, buf, seed, step, nb, r, off, mask_d) == 0
    assert torch.equal(buf, first), "a second call on the same input differs"
    return views, was


@pytest.mark.parametrize("row", GEOMETRY, ids=[geometry_id(r) for r in GEOMETRY])
def test_kernel_matches_the_reference_operation(row, map_dir):
    mp, N, M, H, W, r, nb, seed, step, off, mask_kind = row
    rng = np.random.default_rng(zlib.crc32(geometry_id(row).encode()))
    env = handle(mp, N, M, H, W, map_dir)
    buf, before, _ = guarded((N, M, CLASSES[mp], H, W), rng)
    mask = make_mask(mask_kind, N, rng)
    views, was = check_call(env, row, mask, buf, before)
    if nb == 0 or mask_kind == "off":
        assert np.array_equal(views, was)
    else:
        assert not np.array_equal(views, was)
    env.close()


def test_kernel_on_a_buffer_beyond_2gb(map_dir):
    """1400 Knuffingen envs at 480x640: 2.15e9 bytes, so the view base (blockIdx.x * C * H * W) passes 2^31; the wrapper's
    defaults (radius 100, 10 blobs); a sample of views that includes the first, the last and those across 2^31 bytes"""
    N, H, W, Cn = 1400, 480, 640, 5
    n = N * Cn * H * W
    assert n > 2**31
    env = handle("knuffingen", N, 1, H, W, map_dir)
    g = torch.Generator(device=DEV).manual_seed(5)
    buf = torch.randint(0, 256, (n + 2 * GUARD,), dtype=torch.uint8, device=DEV, generator=g)
    before = buf.clone()
    assert noise(env, buf, 0x1234567890, 3, 10, 100, 0) == 0
    assert torch.equal(buf[:GUARD], before[:GUARD]) and torch.equal(buf[GUARD + n:], before[GUARD + n:]), "guard band written"
    per = Cn * H * W
    cross = (2**31) // per
    sample = sorted({0, 1, cross - 1, cross, cross + 1, N - 2, N - 1} | set(np.random.default_rng(3).integers(0, N, 8).tolist()))
    views, was = buf[GUARD:GUARD + n].view(N, 1, Cn, H, W), before[GUARD:GUARD + n].view(N, 1, Cn, H, W)
    for i in sample:
        want = reference_noise(was[i, 0].cpu().numpy(), i, 0, 0x1234567890, 3, 10, 100)
        assert np.array_equal(views[i, 0].cpu().numpy(), want), ("env", i)
    first = buf.clone()
    buf.copy_(before)
    assert noise(env, buf, 0x1234567890, 3, 10, 100, 0) == 0
    assert torch.equal(buf, first), "a second call on the same input differs"
    del buf, before, first
    env.close()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("max_radius,n_blobs", [(0, 10), (1024, 10), (100, -1)])
def test_invalid_arguments_leave_the_buffer_untouched(max_radius, n_blobs, map_dir):
    rng = np.random.default_rng(max_radius)
    env = handle("knuffingen", 4, 1, 45, 71, map_dir)
    buf, before, _ = guarded((4, 1, 5, 45, 71), rng)
    assert noise(env, buf, 1, 0, n_blobs, max_radius, 0) == TC_ERR_INVALID
    assert np.array_equal(buf.cpu().numpy(), before)
    env.close()


def actions(rng, n):
    cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
    return {"car_control": torch.from_numpy(cc).to(DEV), "maneuver": torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)).to(DEV)}


@pytest.mark.parametrize("res,max_radius,n_blobs", [([128, 160], 100, 10), ([84, 84], 30, 6), ([96, 128], 2, 3)])
def test_noise_wrapper_matches_the_reference_operation(res, max_radius, n_blobs):
    from tinycarlo_b200 import TinyCarloVecEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    n, seed, off = 48, 0x1234567890, 1000
    cfg = make_config("knuffingen", "classes", cam={"resolution": res})
    base = TinyCarloVecEnv(cfg, n, device="cuda:0", env_index_offset=off)
    clean = TinyCarloVecEnv(cfg, n, device="cuda:0", env_index_offset=off)
    env = NoiseObservationWrapper(base, blob_max_radius=max_radius, n_blobs=n_blobs, seed=seed)
    assert base.wrapped
    env.reset(seed=1)
    clean.reset(seed=1)
    rng = np.random.default_rng(0)
    changed = 0
    for t in range(4):
        act = {"car_control": torch.from_numpy(np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)).cuda(),
               "maneuver": torch.zeros(n, dtype=torch.int32, device="cuda")}
        obs, *_ = env.step(act)
        cobs, *_ = clean.step(act)
        got, c = obs.cpu().numpy(), cobs.cpu().numpy()
        for i in range(n):
            want = reference_noise(c[i].copy(), off + i, 0, seed, t, n_blobs, max_radius)
            assert np.array_equal(got[i], want), (t, i)
        changed += int((got != c).sum())
    assert changed > 0
    base.close()
    clean.close()


def test_wrapper_rollout_at_480x640_with_autoresets():
    """default wrapper arguments on the headline frame; envs marked done are reset by the next step, and those spawn frames
    are noised too (with that step's counter)"""
    from tinycarlo_b200 import TinyCarloVecEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    n, off, seed = 12, 300, 0xFFFFFFFF00000000
    cfg = make_config("knuffingen", "classes", cam={"resolution": [480, 640]})
    base = TinyCarloVecEnv(cfg, n, device=DEV, env_index_offset=off, autoreset="next_step")
    clean = TinyCarloVecEnv(cfg, n, device=DEV, env_index_offset=off, autoreset="next_step")
    env = NoiseObservationWrapper(base, seed=seed)
    assert (env.max_radius, env.n_blobs) == (100, 10)
    clean.set_wrapped(True)
    env.reset(seed=4)
    clean.reset(seed=4)
    rng = np.random.default_rng(4)
    resets = 0
    for t in range(6):
        act = actions(rng, n)
        obs = env.step(act)[0].cpu().numpy()
        cobs = clean.step(act)[0].cpu().numpy()
        assert torch.equal(base.reset_mask, clean.reset_mask)
        resets += int(clean.reset_mask.sum())
        for i in range(n):
            assert np.array_equal(obs[i], reference_noise(cobs[i].copy(), off + i, 0, seed, t, 10, 100)), (t, i)
        done = torch.from_numpy(rng.random(n) < 0.3).to(DEV)
        base.mark_done(done)
        clean.mark_done(done)
    assert resets > 0
    base.close()
    clean.close()


def test_noise_wrapper_on_the_single_env_drop_in():
    """several steps of the drop-in against a clean twin through the reference"""
    from tinycarlo_b200 import TinyCarloEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    cfg = make_config("knuffingen", "classes")
    env = NoiseObservationWrapper(TinyCarloEnv(config=cfg), blob_max_radius=60, n_blobs=8, seed=5)
    clean = TinyCarloEnv(config=cfg)
    clean.wrapped = True
    env.reset(seed=0)
    clean.reset(seed=0)
    for t in range(5):
        act = {"car_control": [0.8, 0.3 * np.sin(t)], "maneuver": t % 3}
        o = env.step(act)[0]
        c = clean.step(act)[0]
        assert o.shape == (5, 128, 160) and set(np.unique(o)).issubset({0, 255})
        assert np.array_equal(o, reference_noise(c.copy(), 0, 0, 5, t, 8, 60)), t
        assert not np.array_equal(o, c)
    env.close()
    clean.close()


@pytest.mark.parametrize("fmt", ["rgb", "classes_bits", "classes_bf16"])
def test_wrapper_leaves_other_formats_unchanged(fmt):
    from tinycarlo_b200 import TinyCarloVecEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    n = 16
    cfg = make_config("knuffingen", "rgb" if fmt == "rgb" else "classes")
    kw = {} if fmt == "rgb" else {"obs_format": fmt}
    base, clean = TinyCarloVecEnv(cfg, n, device=DEV, **kw), TinyCarloVecEnv(cfg, n, device=DEV, **kw)
    env = NoiseObservationWrapper(base, seed=3)
    clean.set_wrapped(True)
    env.reset(seed=2)
    clean.reset(seed=2)
    rng = np.random.default_rng(2)
    for t in range(3):
        act = actions(rng, n)
        o, c = env.step(act)[0], clean.step(act)[0]
        assert o.dtype == c.dtype and torch.equal(o, c), t
    base.close()
    clean.close()


GROUPS = [(5, [84, 84]), (7, [128, 160]), (4, [45, 71])]


def grouped_rollout(groups, env_index_offset=0, group_index_offsets=None, seed=0x5EED):
    """a grouped env (Knuffingen, the given groups) under the noise wrapper, reset"""
    from tinycarlo_b200 import TinyCarloGroupedVecEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    cfg = make_config("knuffingen", "classes")
    g = TinyCarloGroupedVecEnv(cfg, groups, device=DEV, env_index_offset=env_index_offset, group_index_offsets=group_index_offsets)
    env = NoiseObservationWrapper(g, blob_max_radius=40, n_blobs=6, seed=seed)
    env.reset(seed=9)
    return g, env


def test_wrapper_on_the_grouped_env():
    """each group is noised with its own handle and env_index_offset: the same as standalone envs at those offsets"""
    from tinycarlo_b200 import TinyCarloVecEnv
    from tinycarlo_b200.wrapper import NoiseObservationWrapper
    off, n = 1000, sum(k for k, _ in GROUPS)
    g, env = grouped_rollout(GROUPS, env_index_offset=off)
    solo, start = [], off
    for k, res in GROUPS:
        e = NoiseObservationWrapper(TinyCarloVecEnv(make_config("knuffingen", "classes", cam={"resolution": res}), k, device=DEV,
                                                    env_index_offset=start), blob_max_radius=40, n_blobs=6, seed=0x5EED)
        e.reset(seed=9)
        solo.append(e)
        start += k
    rng = np.random.default_rng(6)
    for t in range(3):
        act = actions(rng, n)
        obs = env.step(act)[0]
        lo = 0
        for (k, _), e, o in zip(GROUPS, solo, obs):
            want = e.step({key: v[lo:lo + k] for key, v in act.items()})[0]
            assert torch.equal(o, want), (t, k)
            lo += k
    g.close()
    for e in solo:
        e.close()


def test_wrapper_on_sharded_groups_equals_the_job():
    """two shards from distributed.shard_groups give, env for env, the noised observations of the unsharded job"""
    from tinycarlo_b200.distributed import shard_groups
    sizes = [k for k, _ in GROUPS]
    job, jenv = grouped_rollout(GROUPS)
    shards = []
    for rank in range(2):
        local, offs = shard_groups(sizes, rank, 2)
        shards.append((local, offs) + grouped_rollout([(k, res) for k, (_, res) in zip(local, GROUPS)], group_index_offsets=offs))
    rng = np.random.default_rng(8)
    starts = np.cumsum([0] + sizes)
    for t in range(3):
        act = actions(rng, sum(sizes))
        jobs = jenv.step(act)[0]
        for local, offs, _, senv in shards:
            idx = np.concatenate([np.arange(o, o + k) for o, k in zip(offs, local)])
            sobs = senv.step({key: v[torch.from_numpy(idx).to(DEV)] for key, v in act.items()})[0]
            for gi, (k, o) in enumerate(zip(local, offs)):
                lo = o - starts[gi]
                assert torch.equal(sobs[gi], jobs[gi][lo:lo + k]), (t, gi)
    job.close()
    for s in shards:
        s[2].close()
