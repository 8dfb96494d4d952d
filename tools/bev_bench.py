"""Speed of the bird's-eye view (config section `bev`, tc_bev_kernel): the kernel alone (render_bev in a loop between CUDA
events; bytes = the BEV frames it writes, against this card's measured device-to-device copy rate) and env-steps/s with the
BEV on and off, the two envs alternated in the same process, on the shapes of bench.py's config 2 (4096 envs, simple_layout
84x84 classes, steps replayed from a CUDA graph) and config 3 (16384 envs, Knuffingen 480x640 classes, eager steps).
Prints the card's name and power limit beside the numbers, and one JSON line at the end.

    python tools/bev_bench.py [--rounds 3] [--steps 50] [--kernel-iters 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tinycarlo_b200 import TinyCarloVecEnv  # noqa: E402
from tinycarlo_b200._lib import build_info  # noqa: E402
from tinycarlo_b200.config import make_config  # noqa: E402

BEV = {"resolution": [128, 128], "route": True, "line_thickness": 1}
SHAPES = [("config2", "simple_layout", [84, 84], 4096, True), ("config3", "knuffingen", [480, 640], 16384, False)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters   # ms per call


def copy_peak_gbs():
    """device-to-device copy of 4 GB (read + write bytes over time): the copy peak the kernel's write rate is set against"""
    a = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    ms = min(timed(lambda: b.copy_(a), 5) for _ in range(3))
    del a, b
    torch.cuda.empty_cache()
    return 2 * (4 << 30) / (ms * 1e-3) / 1e9


def make_env(map_name, res, n, bev):
    cfg = make_config(map_name, "classes", cam={"resolution": res})
    if bev:
        cfg["bev"] = dict(BEV)
    env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    env.reset(seed=0)
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--kernel-iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bev_bench.py needs a CUDA device")
    name = card()
    peak = copy_peak_gbs()
    print(f"card: {name} (name, power limit, max SM clock); library {build_info()}")
    print(f"device-to-device copy peak: {peak:.0f} GB/s")
    result = {"card": name, "copy_peak_gbs": peak, "bev": BEV, "shapes": {}}
    for label, map_name, res, n, graph in SHAPES:
        rng = np.random.default_rng(0)
        cc = torch.from_numpy(np.stack([rng.uniform(0.2, 1.0, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)).cuda()
        man = torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)).cuda()
        action = {"car_control": cc, "maneuver": man}
        envs = {"off": make_env(map_name, res, n, False), "on": make_env(map_name, res, n, True)}
        on = envs["on"]
        bev_bytes = on.bev.numel() * on.bev.element_size()
        k_ms = min(timed(on.render_bev, args.kernel_iters) for _ in range(3))
        runners = {}
        for key, e in envs.items():
            if graph:
                g = e.capture(lambda _e: action, steps=10, warmup=3)
                runners[key] = (g.replay, 10)
            else:
                runners[key] = ((lambda e=e: e.step(action)), 1)
        rates = {"off": [], "on": []}
        for _ in range(args.rounds):
            for key in ("off", "on"):
                fn, per = runners[key]
                reps = max(args.steps // per, 1)
                ms = timed(fn, reps)
                rates[key].append(n * per / (ms * 1e-3))
        achieved = bev_bytes / (k_ms * 1e-3) / 1e9
        r = {"envs": n, "camera": res, "map": map_name, "graph": graph, "bev_bytes_per_launch": bev_bytes, "bev_kernel_ms": k_ms,
             "bev_kernel_gbs": achieved, "bev_kernel_fraction_of_copy_peak": achieved / peak,
             "env_steps_per_s_off": rates["off"], "env_steps_per_s_on": rates["on"]}
        result["shapes"][label] = r
        print(f"{label}: {n} envs, {map_name} {res[0]}x{res[1]} camera, BEV {BEV['resolution'][0]}x{BEV['resolution'][1]} x {on.bev.shape[1]} planes u8"
              f" | BEV kernel {k_ms:.4f} ms = {achieved:.0f} GB/s = {achieved / peak:.3f} of the copy peak"
              f" | env-steps/s BEV off {', '.join(f'{v / 1e6:.3f}' for v in rates['off'])} M,"
              f" on {', '.join(f'{v / 1e6:.3f}' for v in rates['on'])} M (rounds alternated)")
        for e in envs.values():
            e.close()
        del envs, on, runners
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        time.sleep(0.1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
