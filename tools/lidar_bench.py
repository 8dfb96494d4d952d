"""Speed of the range scan (config section `lidar`, tc_lidar_kernel): the kernel alone (render_lidar in a loop between CUDA
events), env-steps/s with the scan on and off, the two envs alternated in the same process, on the shapes of bench.py's
config 2 (4096 envs, simple_layout 84x84 classes, steps replayed from a CUDA graph) and config 3 (16384 envs, Knuffingen
480x640 classes, eager steps), and a scan-only rollout (no_observation: the tracking kernel and the scan) on Knuffingen at
32768 envs, graph-replayed, against the same rollout without the scan. Prints the card's name and power limit beside the
numbers, and one JSON line at the end.

    python tools/lidar_bench.py [--rounds 3] [--steps 50] [--kernel-iters 200]
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

LIDAR = {"rays": 64, "fov": 360, "max_range": 0.5}
# (label, map, camera resolution, envs, graph-replayed, no_observation)
SHAPES = [("config2", "simple_layout", [84, 84], 4096, True, False), ("config3", "knuffingen", [480, 640], 16384, False, False),
          ("scan_only", "knuffingen", [84, 84], 32768, True, True)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
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


def make_env(map_name, res, n, lidar, no_obs):
    cfg = make_config(map_name, "classes", cam={"resolution": res})
    if lidar:
        cfg["lidar"] = dict(LIDAR)
    env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    env.no_observation = no_obs
    env.reset(seed=0)
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--kernel-iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lidar_bench.py needs a CUDA device")
    name = card()
    print(f"card: {name} (name, power limit); library {build_info()}")
    result = {"card": name, "lidar": LIDAR, "shapes": {}}
    for label, map_name, res, n, graph, no_obs in SHAPES:
        rng = np.random.default_rng(0)
        cc = torch.from_numpy(np.stack([rng.uniform(0.2, 1.0, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)).cuda()
        man = torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)).cuda()
        action = {"car_control": cc, "maneuver": man}
        envs = {"off": make_env(map_name, res, n, False, no_obs), "on": make_env(map_name, res, n, True, no_obs)}
        on = envs["on"]
        k_ms = min(timed(on.render_lidar, args.kernel_iters) for _ in range(3))
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
                ms = timed(fn, max(args.steps // per, 1))
                rates[key].append(n * per / (ms * 1e-3))
        hits = float((on.lidar < LIDAR["max_range"]).float().mean().item())
        r = {"envs": n, "camera": None if no_obs else res, "map": map_name, "graph": graph, "no_observation": no_obs,
             "lidar_kernel_ms": k_ms, "lidar_bytes_per_env": on.lidar[0].numel() * 4, "fraction_of_rays_with_a_hit": hits,
             "env_steps_per_s_off": rates["off"], "env_steps_per_s_on": rates["on"]}
        result["shapes"][label] = r
        print(f"{label}: {n} envs, {map_name} " + ("no observation" if no_obs else f"{res[0]}x{res[1]} camera")
              + f", scan {LIDAR['rays']} rays x {on.lidar.shape[1]} classes | kernel {k_ms:.4f} ms"
              f" | env-steps/s scan off {', '.join(f'{v / 1e6:.3f}' for v in rates['off'])} M,"
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
