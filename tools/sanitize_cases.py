"""A small pass through every kernel of the library for compute-sanitizer (memcheck / racecheck / initcheck / synccheck): few envs
(except where the thread-per-env tracking kernel needs many), few steps, each render path once - the packed and one-env
block-per-env kernels, the per-class headline kernel, the banded kernel (RGB), the two-kernel path of bit-packed frames with its
overflow fallback, the unfused debug path, both tracking kernels (warp- and thread-per-env, chosen by the env count) incl. u-turn
scans and in-kernel autoreset, the noise kernel - every frame compared with the CPU oracle.

  compute-sanitizer --tool racecheck python tools/sanitize_cases.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from pair_util import make_config, oracle_env  # noqa: E402
from tinycarlo_b200 import TinyCarloVecEnv  # noqa: E402

STEPS = int(os.environ.get("TC_SAN_STEPS", 3))
# tc_create's choice of tracking kernel: one thread per env once n / 4 > 3 * 8 * SMs, below that a warp per env (8 lanes per env
# above 3 * 8 * SMs / 2 envs)
SMS = torch.cuda.get_device_properties(0).multi_processor_count
N_THREAD_TRACK = 4 * (3 * 8 * SMS + 1)


def run(name, cfg, n, env_kw=None, setenv=None, check="u8"):
    old = {k: os.environ.get(k) for k in (setenv or {})}
    os.environ.update(setenv or {})
    try:
        env = TinyCarloVecEnv(cfg, n, device="cuda:0", **(env_kw or {}))
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
    ocfg = dict(cfg, sim=dict(cfg["sim"]))
    oenv = oracle_env(ocfg, n)
    rng = np.random.default_rng(7)
    env.reset(seed=5)
    oenv.reset(env._spawn_nodes.cpu().numpy())
    H, W = cfg["camera"]["resolution"]

    def same():
        o = env.obs.cpu().numpy()
        if check == "bits":
            o = np.unpackbits(o.view(np.uint32).view(np.uint8), axis=-1, bitorder="little")[..., : H * W].reshape(n, -1, H, W) * 255
        return np.array_equal(o, oenv.obs)
    assert same(), name + ": reset frames"
    for t in range(STEPS):
        cc = np.stack([rng.uniform(0.3, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)
        man = rng.integers(0, 4, n).astype(np.int32)
        env.step({"car_control": torch.from_numpy(cc).cuda(), "maneuver": torch.from_numpy(man).cuda()})
        oenv.step(cc.astype(np.float64), man)
        done = (oenv.terminated | oenv.truncated).astype(bool)
        assert same(), f"{name}: frames at step {t}"
        if env.autoreset:
            break   # one autoreset-enabled step is enough here (the flags path); the parity tests cover the rest
        if done.any():
            env.reset_done()
            oenv.reset(env._spawn_nodes.cpu().numpy(), mask=done)
    torch.cuda.synchronize()
    info = env.render_info()
    env.close()
    print(f"ok  {name:44s} {info}", flush=True)


knuff = lambda fmt, res, **cam: make_config("knuffingen", fmt, cam=dict(resolution=res, **cam))  # noqa: E731
simple = lambda fmt, res, **cam: make_config("simple_layout", fmt, cam=dict(resolution=res, **cam), car={"max_velocity": 0.15})  # noqa: E731
run("packed env kernel 128x160 (2 envs/block)", knuff("classes", [128, 160]), 13)
run("one-env kernel 128x160", knuff("classes", [128, 160]), 9, setenv={"TC_ENV_PACK": "0"})
run("packed env kernel 84x84, 2 chunks", simple("classes", [84, 84]), 12)
run("packed env kernel rgb 96x128", simple("rgb", [96, 128]), 7)
run("env kernel 240x320", knuff("classes", [240, 320]), 5)
run("per-class headline kernel 480x640", knuff("classes", [480, 640]), 3)
run("banded kernel rgb 480x640", simple("rgb", [480, 640]), 3)
run("bits 480x640: prims + draw kernels", knuff("classes", [480, 640]), 4, env_kw={"obs_format": "classes_bits"}, check="bits")
run("bits 480x640 long range: overflow fallback", simple("classes", [480, 640], max_range=3.0, orientation=[30, 0, 0]), 3,
    env_kw={"obs_format": "classes_bits"}, check="bits")
run("unfused project + raster (debug segments)", knuff("classes", [96, 128]), 4, env_kw={"debug_segments": True})
run("thread-per-env tracking", knuff("classes", [32, 48]), N_THREAD_TRACK)
run("warp-per-env tracking", knuff("classes", [32, 48]), 20)
run("autoreset next_step (thread tracking)", knuff("classes", [32, 48]), N_THREAD_TRACK, env_kw={"autoreset": "next_step"})
# the noise kernel (NoiseObservationWrapper on the device)
from tinycarlo_b200.wrapper import NoiseObservationWrapper  # noqa: E402
e = TinyCarloVecEnv(knuff("classes", [64, 96]), 6, device="cuda:0")
w = NoiseObservationWrapper(e, blob_max_radius=9, n_blobs=4)
w.reset(seed=1)
w.step({"car_control": torch.zeros((6, 2), device="cuda"), "maneuver": torch.zeros(6, dtype=torch.int32, device="cuda")})
torch.cuda.synchronize()
e.close()
print("ok  noise kernel", flush=True)
print("sanitize_cases: all paths ran and matched the oracle")
