"""Speed of the navigation goals (config section `navigation`, tc_route_kernel): the kernel alone at 4096, 16384 and 32768
Knuffingen envs (tc_update_route between CUDA events, once recomputing at the current goals and once drawing new ones), and
env-steps/s with the section on and off, the two envs alternated in the same process, on the shapes of bench.py's config 2
(4096 envs, simple_layout 84x84 classes, steps replayed from a CUDA graph) and config 3 (16384 envs, Knuffingen 480x640
classes, eager steps). Prints the card's name and power limit beside the numbers, and one JSON line at the end.

    python tools/route_bench.py [--rounds 3] [--steps 50] [--kernel-iters 500]
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

KERNEL_ENVS = [4096, 16384, 32768]
# (label, map, camera resolution, envs, graph-replayed)
SHAPES = [("config2", "simple_layout", [84, 84], 4096, True), ("config3", "knuffingen", [480, 640], 16384, False)]


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


def make_env(map_name, res, n, nav, no_obs=False):
    cfg = make_config(map_name, "classes", cam={"resolution": res})
    if nav:
        cfg["navigation"] = {}
    env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    env.no_observation = no_obs
    env.reset(seed=0)
    return env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--kernel-iters", type=int, default=500)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("route_bench.py needs a CUDA device")
    name = card()
    print(f"card: {name} (name, power limit); library {build_info()}")
    result = {"card": name, "kernel": {}, "shapes": {}}
    for n in KERNEL_ENVS:
        env = make_env("knuffingen", [84, 84], n, True, no_obs=True)
        rec = min(timed(lambda: env._update_route(None, draw=False), args.kernel_iters) for _ in range(3))
        drw = min(timed(lambda: env._update_route(None, draw=True), args.kernel_iters) for _ in range(3))
        result["kernel"][n] = {"recompute_ms": rec, "draw_ms": drw, "goals": len(env.nav_cfg["goals"])}
        print(f"tc_route_kernel at {n} envs ({len(env.nav_cfg['goals'])} goals): {rec * 1e3:.2f} us recomputing, "
              f"{drw * 1e3:.2f} us drawing every env")
        env.close()
    for label, map_name, res, n, graph in SHAPES:
        rng = np.random.default_rng(0)
        cc = torch.from_numpy(np.stack([rng.uniform(0.2, 1.0, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)).cuda()
        man = torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)).cuda()
        action = {"car_control": cc, "maneuver": man}
        envs = {"off": make_env(map_name, res, n, False), "on": make_env(map_name, res, n, True)}
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
        result["shapes"][label] = {"envs": n, "camera": res, "map": map_name, "graph": graph, "env_steps_per_s_off": rates["off"],
                                   "env_steps_per_s_on": rates["on"]}
        print(f"{label}: {n} envs, {map_name} {res[0]}x{res[1]} | env-steps/s navigation off "
              f"{', '.join(f'{v / 1e6:.3f}' for v in rates['off'])} M, on {', '.join(f'{v / 1e6:.3f}' for v in rates['on'])} M"
              " (rounds alternated)")
        for e in envs.values():
            e.close()
        del envs, runners
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        time.sleep(0.1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
