"""Tracked observation buffers (tc_track_obs): the per-class kernel stores only the 32-byte sectors of a 480x640 class mask that
hold a set pixel now or did after the previous render. The frames must stay byte for byte what an untracked render writes, and
every write into the buffer that the renders did not make - seen by torch, declared with invalidate_obs(), or made by the
library through a path that does not keep the mask - must be undone by the next render."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import oracle as orc
from pair_util import make_config
from rig_util import REAR, oracle_views

H, W = 480, 640


def _cfg(**kw):
    return make_config("knuffingen", "classes", cam={"resolution": [H, W]}, **kw)


@functools.lru_cache(maxsize=None)
def _omap(name, ppm, spawn):
    return orc.load_named_map(name, ppm, None if spawn is None else list(spawn))


def oracle_obs(env):
    """the oracle's frames of every view at the env's current state, shaped like env.obs"""
    m = env.config["map"]
    sp = m.get("spawn_points")
    omap = _omap(m["map_name"], m["pixel_per_meter"], None if sp is None else tuple(sp))
    sf = env.state_dict()["sf"].cpu().numpy()
    return oracle_views(omap, env._cam_rows, env._thickness, sf, env.n_cameras, env.H, env.W, "classes").reshape(env.obs.shape)


def untrack(env):
    """a plain handle: tracking switched off, every render stores every byte"""
    env._untrack_obs()
    assert env.obs_mask_words() == 0


def stanley(env, man):
    import torch
    o = env.out
    steer = (o["heading_error"] + torch.atan2(4.0 * o["cte"], torch.full_like(o["cte"], 0.8))) * (180.0 / np.pi / 30.0)
    return {"car_control": torch.stack([torch.full_like(steer, 0.8), steer.clamp(-1, 1)], 1).contiguous(), "maneuver": man}


def _cudart():
    for name in ("libcudart.so", "libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
        try:
            rt = C.CDLL(name)
            rt.cudaMemsetAsync.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]
            return rt
        except OSError:
            continue
    pytest.skip("libcudart not found")


# ------------------------------------------------------------------------------------------------ no GPU needed
def test_entry_points_reject_a_null_handle():
    from tinycarlo_b200 import _lib
    L = _lib.lib()
    assert L.tc_track_obs(None, None) == -1 and b"null handle" in L.tc_last_error()
    assert L.tc_invalidate_obs(None, None) == -1 and b"null handle" in L.tc_last_error()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_tracked_rollout_matches_untracked_and_oracle():
    """257 envs x 150 steps with maneuver changes and next-step autoresets: the tracked frames equal an untracked handle's at
    every step and the oracle's every 10 steps"""
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    n = 257
    a = TinyCarloVecEnv(_cfg(), n, device="cuda:0", autoreset="next_step")
    b = TinyCarloVecEnv(_cfg(), n, device="cuda:0", autoreset="next_step")
    untrack(b)
    a.reset(seed=5)
    b.reset(seed=5)
    assert torch.equal(a.obs, b.obs)
    assert np.array_equal(a.obs.cpu().numpy(), oracle_obs(a)), "reset frames"
    rng = np.random.default_rng(3)
    man = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    resets = 0
    for t in range(150):
        if t % 25 == 0:
            man.copy_(torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)))
        act = stanley(a, man)
        a.step(act)
        b.step(act)
        resets += int(a.reset_mask.sum())
        assert torch.equal(a.obs, b.obs), f"tracked and untracked frames differ at step {t}"
        if t % 10 == 9:
            assert np.array_equal(a.obs.cpu().numpy(), oracle_obs(a)), f"frames differ from the oracle at step {t}"
    assert resets > 0, "the rollout should exercise autoresets"
    assert a.obs.any()


CASES = ["torch_byte", "raw_memset", "noise", "masked_reset", "masked_render", "restore", "replace_obs", "segment_export", "capture"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_the_next_frame_undoes_outside_writes(case):
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv, _lib
    n = 9
    env = TinyCarloVecEnv(_cfg(), n, device="cuda:0", autoreset="next_step")
    env.reset(seed=2)
    man = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    for _ in range(3):
        env.step(stanley(env, man))
    assert env._obs_seen[0] == env.obs.data_ptr()
    hw = H * W
    # class 4 of Knuffingen is never drawn at this camera: its planes are zero and their sectors clean after a render
    plane4 = env.obs[:, 4].reshape(n, -1)
    assert not plane4.any()

    def check(what):
        assert np.array_equal(env.obs.cpu().numpy(), oracle_obs(env)), f"{case}: {what}"

    if case == "torch_byte":
        env.obs[3, 4, 100, 200] = 255
        env.step(stanley(env, man))
        check("after a torch write into a zero sector")
    elif case == "raw_memset":
        rt = _cudart()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        ptr = env.obs.data_ptr() + (2 * 5 + 4) * hw + 4096
        assert rt.cudaMemsetAsync(ptr, 0x7F, 1024, stream) == 0
        env.step(stanley(env, man))
        # torch did not see the write and nobody declared it: the tracked render leaves those clean sectors alone
        assert (env.obs[2, 4].reshape(-1)[4096:4096 + 1024] == 0x7F).all(), "the render should not have stored clean sectors"
        assert rt.cudaMemsetAsync(ptr, 0x7F, 1024, stream) == 0
        env.invalidate_obs()
        env.step(stanley(env, man))
        check("after a raw memset and invalidate_obs()")
    elif case == "noise":
        from tinycarlo_b200.wrapper import NoiseObservationWrapper
        wenv = NoiseObservationWrapper(env, blob_max_radius=60, n_blobs=10, seed=4)
        before = env.obs.clone()
        wenv.step(stanley(env, man))
        assert not torch.equal(env.obs, before)
        env.step(stanley(env, man))
        check("after the noise wrapper")
    elif case == "masked_reset":
        mask = torch.zeros(n, dtype=torch.bool, device="cuda:0")
        mask[::2] = True
        env.obs[1::2, 4].fill_(9)   # envs the reset does not render: the next step must still clean them
        env.reset(mask=mask)
        sel = mask.cpu().numpy()
        assert np.array_equal(env.obs.cpu().numpy()[sel], oracle_obs(env)[sel]), "masked reset"
        env.step(stanley(env, man))
        check("after a masked reset")
    elif case == "masked_render":
        mask = torch.zeros(n, dtype=torch.bool, device="cuda:0")
        mask[1::3] = True
        st = env.state_dict()
        env.step(stanley(env, man))
        env.load_state_dict(st)
        env.render_obs(mask)           # the selected envs go back a step, the others keep the newer frame
        env.render_obs()
        check("after a masked render_obs")
    elif case == "restore":
        ck = env.checkpoint()
        for _ in range(4):
            env.step(stanley(env, man))
        env.restore(ck)
        check("after restore()")
        env.step(stanley(env, man))
        check("the step after restore()")
    elif case == "replace_obs":
        old = env.obs
        env.obs = torch.full_like(old, 0xAB)
        env._outs = env._make_outputs(with_obs=True)
        env.step(stanley(env, man))
        assert env._obs_seen[0] == env.obs.data_ptr()
        check("after replacing env.obs")
        env.render_obs()
        check("render_obs into the new tensor")
    elif case == "segment_export":
        st = env.state_dict()
        other = {k: v.roll(1, 0).contiguous() for k, v in st.items()}
        V = n * env.n_cameras
        cnt = torch.zeros((V, env.n_classes), dtype=torch.int32, device="cuda:0")
        seg = torch.zeros((V, int(env.map.ll_edge_off[-1]), 4), dtype=torch.int32, device="cuda:0")
        env.load_state_dict(other)
        # the unfused path with segment export draws other poses into the tracked buffer without keeping the mask
        _lib.check(env._L.tc_render(env._h, None, C.c_void_p(env.obs.data_ptr()), _lib.TC_OBS_CLASSES, C.c_void_p(cnt.data_ptr()),
                                    C.c_void_p(seg.data_ptr()), env._stream()), "tc_render")
        check("the segment-export render itself")
        env.load_state_dict(st)
        env.render_obs()
        check("the tracked render after a segment-export render")
    elif case == "capture":
        act = stanley(env, man)
        g = env.capture(lambda e: act, steps=1)
        assert not env._track_obs
        g.replay()
        env.obs[5, 4, 10:20, 30:40] = 77
        g.replay()
        torch.cuda.synchronize()
        check("after a graph replay that followed a torch write")


@pytest.mark.gpu
def test_two_camera_rig_at_480x640():
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    cfg = _cfg()
    cfg["cameras"] = [{}, REAR]
    n = 7
    a = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    b = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    untrack(b)
    a.reset(seed=9)
    b.reset(seed=9)
    man = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    for t in range(12):
        act = stanley(a, man)
        a.step(act)
        b.step(act)
        assert torch.equal(a.obs, b.obs), f"step {t}"
    assert a.obs.shape == (n, 2, a.n_classes, H, W)
    assert np.array_equal(a.obs.cpu().numpy(), oracle_obs(a))


@pytest.mark.gpu
def test_untracked_handle_overwrites_a_poisoned_buffer():
    """without tc_track_obs the per-class kernel stores every byte, as before"""
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    n = 6
    env = TinyCarloVecEnv(_cfg(), n, device="cuda:0")
    untrack(env)
    env.obs.fill_(0xAB)
    env.reset(seed=1)
    assert np.array_equal(env.obs.cpu().numpy(), oracle_obs(env))
    man = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    for _ in range(3):
        env.obs.fill_(0xAB)
        env.step(stanley(env, man))
        assert np.array_equal(env.obs.cpu().numpy(), oracle_obs(env))


@pytest.mark.gpu
def test_track_obs_argument_validation():
    from tinycarlo_b200 import TinyCarloVecEnv
    env = TinyCarloVecEnv(_cfg(), 3, device="cuda:0")
    L, h = env._L, env._h
    p = env.obs.data_ptr()
    assert L.tc_track_obs(h, C.c_void_p(p + 16)) == -1 and b"32-byte aligned" in L.tc_last_error()
    assert L.tc_track_obs(h, C.c_void_p(p)) == 0
    assert env.obs_mask_words() == 3 * env.n_classes * (H * W // 1024)
    assert L.tc_invalidate_obs(h, None) == 0
    assert L.tc_track_obs(h, None) == 0
    assert env.obs_mask_words() == 0
    assert L.tc_invalidate_obs(h, None) == 0   # nothing tracked: nothing to do
    assert L.tc_obs_mask(h, None, None, None) == -1
    bits = TinyCarloVecEnv(_cfg(), 3, device="cuda:0", obs_format="classes_bits")
    assert not bits._track_obs
    assert bits._L.tc_track_obs(bits._h, C.c_void_p(bits.obs.data_ptr())) == -1 and b"TC_OBS_CLASSES" in bits._L.tc_last_error()
    assert bits._L.tc_track_obs(bits._h, None) == 0


def _sector_mask(obs):
    """the exact mask of a u8 buffer [V,C,H,W]: bit b of word w of a plane = sector 32w+b holds a non-zero byte"""
    nz = (obs.reshape(-1, H * W // 32, 32) != 0).any(axis=2)
    return np.packbits(nz, axis=1, bitorder="little").view(np.uint32).reshape(-1)


@pytest.mark.gpu
def test_the_mask_is_exact_after_every_render():
    """after each tracked render the mask words are exactly the sectors that hold a set pixel, so a step stores the sectors
    non-zero in the previous frame or in this one and no others"""
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    n = 11
    env = TinyCarloVecEnv(_cfg(), n, device="cuda:0", autoreset="next_step")
    words = env.obs_mask_words()
    assert words == n * env.n_classes * (H * W // 1024)
    m = torch.zeros(words, dtype=torch.int32, device="cuda:0")
    env.reset(seed=3)
    man = torch.ones(n, dtype=torch.int32, device="cuda:0")
    for t in range(8):
        env.obs_mask_words(m)
        assert np.array_equal(m.cpu().numpy().view(np.uint32), _sector_mask(env.obs.cpu().numpy())), f"mask after render {t}"
        env.step(stanley(env, man))
    env.obs[0, 0, 0, 0] = 1        # seen by torch: the next step starts from an all-dirty mask
    env.step(stanley(env, man))
    env.obs_mask_words(m)
    assert np.array_equal(m.cpu().numpy().view(np.uint32), _sector_mask(env.obs.cpu().numpy()))


@pytest.mark.gpu
@pytest.mark.parametrize("res", [[84, 84], [H, W]], ids=["84x84", "480x640"])
def test_env_built_and_stepped_in_inference_mode(res):
    """an inference tensor has no version counter: such an env is never tracked and renders whole frames"""
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    n = 5
    cfg = make_config("knuffingen", "classes", cam={"resolution": res})
    with torch.inference_mode():
        env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
        assert env.obs.is_inference() and not env._track_obs and env.obs_mask_words() == 0
        env.reset(seed=4)
        man = torch.zeros(n, dtype=torch.int32, device="cuda:0")
        for _ in range(3):
            env.obs.fill_(0xAB)
            env.step(stanley(env, man))
            assert np.array_equal(env.obs.cpu().numpy(), oracle_obs(env))
    # a tracked env whose tensor is replaced by an inference tensor stops tracking at the next call
    env = TinyCarloVecEnv(_cfg(), n, device="cuda:0")
    assert env._track_obs
    with torch.inference_mode():
        inf = torch.full_like(env.obs, 0xAB)
    env.obs = inf
    env.render_obs()
    assert not env._track_obs and env.obs_mask_words() == 0
    assert np.array_equal(env.obs.cpu().numpy(), oracle_obs(env))


@pytest.mark.gpu
def test_small_frames_keep_no_mask():
    from tinycarlo_b200 import TinyCarloVecEnv
    env = TinyCarloVecEnv(make_config("knuffingen", "classes", cam={"resolution": [128, 160]}), 4, device="cuda:0")
    assert not env._track_obs and env.obs_mask_words() == 0


@pytest.mark.gpu
def test_hand_captured_graph_switches_tracking_off():
    """a rollout captured with torch.cuda.graph directly: the step inside the capture switches tracking off, so a torch write
    between replays is overwritten by the next replay"""
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    n = 6
    env = TinyCarloVecEnv(_cfg(), n, device="cuda:0", autoreset="next_step")
    env.reset(seed=6)
    man = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    act = stanley(env, man)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        env.step(act)
    torch.cuda.current_stream().wait_stream(side)
    assert env._track_obs
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.step(act)
    assert not env._track_obs and env.obs_mask_words() == 0
    g.replay()
    env.obs[2, 4, 50:60, 70:90] = 99
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(env.obs.cpu().numpy(), oracle_obs(env))
