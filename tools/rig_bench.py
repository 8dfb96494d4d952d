"""Speed of camera rigs (the config's `cameras` list, tc_create_rig): M = 1, 2 and 4 cameras per car on three shapes -
bench.py's config 2 (simple_layout 84x84 classes, 4096 envs, eager and replayed from a CUDA graph), Knuffingen 128x160
classes with 32768 envs, and config 3 (Knuffingen 480x640 classes, 16384 envs).

For each shape and M it reports env-steps/s and view-steps/s of the rig, the tracking and render milliseconds per step from
profile_begin / profile_end, and the render milliseconds of a flat one-camera handle of N*M envs with the same camera rows,
whose cars are driven with each rig car's actions M times (so its frames are the rig's views). Rig and flat runs alternate,
and each env is freed before the next is built. Where N*M frames would not fit the card the env count is lowered and the
line says so. Prints the card's name and power limit beside the numbers, and one JSON line at the end.

    python tools/rig_bench.py [--rounds 2] [--steps 20] [--cameras 1 2 4]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tinycarlo_b200 import TinyCarloVecEnv  # noqa: E402
from tinycarlo_b200._lib import build_info  # noqa: E402
from tinycarlo_b200.config import make_config  # noqa: E402

# the rig's cameras in order: the config's camera, a rear camera, a wide one, a side one
CAMERAS = [{}, {"orientation": [22, 0, 180]}, {"fov": 110}, {"orientation": [22, 0, 90]}]
# label, map, camera resolution, envs, steps replayed from a CUDA graph
SHAPES = [("config2_eager", "simple_layout", [84, 84], 4096, False), ("config2_graph", "simple_layout", [84, 84], 4096, True),
          ("knuff_128x160", "knuffingen", [128, 160], 32768, False), ("config3", "knuffingen", [480, 640], 16384, False)]
OBS_BUDGET = 120e9   # bytes of frames one env may hold next to the rest on a 180 GB card


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


def free(*envs):
    for e in envs:
        e.close()
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def profiled(env, action, steps):
    """tracking and render (camera pass + raster) milliseconds per eager step"""
    env.profile_begin(steps)
    for _ in range(steps):
        env.step(action)
    ms, k = env.profile_end()
    return ms["track"] / k, (ms["project"] + ms["raster"]) / k


def run_rig(map_name, res, n, m, graph, action, steps):
    cfg = make_config(map_name, "classes", cam={"resolution": res})
    cfg["cameras"] = CAMERAS[:m]
    env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step")
    env.reset(seed=0)
    spawn = env._spawn_nodes.clone()
    for _ in range(3):
        env.step(action)
    track_ms, render_ms = profiled(env, action, steps)
    if graph:
        g = env.capture(lambda _e: action, steps=10, warmup=3)
        ms = timed(g.replay, max(steps // 10, 1)) / 10
    else:
        ms = timed(lambda: env.step(action), steps)
    rows, thick = env._cam_rows.copy(), env._thickness.copy()
    free(env)
    return {"env_steps_per_s": n / (ms * 1e-3), "view_steps_per_s": n * m / (ms * 1e-3), "step_ms": ms, "track_ms": track_ms,
            "render_ms": render_ms}, (rows, thick, spawn)


def run_flat(map_name, res, n, m, action, like, steps):
    """one camera per env, N*M envs with the rig's rows; car k*M + j starts on rig car k's spawn node and gets its actions
    (after an autoreset the spawn draws differ, which moves a few cars elsewhere on the map)"""
    rows, thick, spawn = like
    cfg = make_config(map_name, "classes", cam={"resolution": res})
    env = TinyCarloVecEnv(cfg, n * m, device="cuda:0", autoreset="next_step")
    env.set_camera_rows(rows, line_thickness=thick)
    env.reset(seed=0, spawn_nodes=spawn.repeat_interleave(m, 0))
    act = {k: v.repeat_interleave(m, 0) for k, v in action.items()}
    for _ in range(3):
        env.step(act)
    track_ms, render_ms = profiled(env, act, steps)
    free(env)
    return {"track_ms": track_ms, "render_ms": render_ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--cameras", type=int, nargs="+", default=[1, 2, 4])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rig_bench.py needs a CUDA device")
    name = card()
    print(f"card: {name} (name, power limit, max SM clock); library {build_info()}", flush=True)
    result = {"card": name, "cameras": CAMERAS, "shapes": {}}
    for label, map_name, res, n0, graph in SHAPES:
        C = 5 if map_name == "knuffingen" else 3
        for m in args.cameras:
            n = n0
            while n * m * C * res[0] * res[1] > OBS_BUDGET:
                n //= 2
            rng = np.random.default_rng(0)
            action = {"car_control": torch.from_numpy(np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n)], 1).astype(np.float32)).cuda(),
                      "maneuver": torch.from_numpy(rng.integers(0, 4, n).astype(np.int32)).cuda()}
            rig, flat = [], []
            for _ in range(args.rounds):   # alternated
                r, like = run_rig(map_name, res, n, m, graph, action, args.steps)
                rig.append(r)
                if not graph:
                    flat.append(run_flat(map_name, res, n, m, action, like, args.steps))
            key = f"{label}_M{m}"
            result["shapes"][key] = {"map": map_name, "camera": res, "envs": n, "envs_asked": n0, "cameras": m, "graph": graph,
                                     "rig": rig, "flat": flat}
            note = "" if n == n0 else f" (lowered from {n0}: {n0 * m} frames would not fit)"
            f = lambda k, rs: ", ".join(f"{x[k]:.4f}" for x in rs)  # noqa: E731
            print(f"{key}: {n} envs{note} x {m} cameras, {map_name} {res[0]}x{res[1]} {'graph' if graph else 'eager'}"
                  f" | M env-steps/s {', '.join(f'{x['env_steps_per_s'] / 1e6:.3f}' for x in rig)}"
                  f" | M view-steps/s {', '.join(f'{x['view_steps_per_s'] / 1e6:.3f}' for x in rig)}"
                  f" | rig track ms {f('track_ms', rig)} render ms {f('render_ms', rig)}"
                  + (f" | flat N*M render ms {f('render_ms', flat)} track ms {f('track_ms', flat)}" if flat else ""), flush=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
