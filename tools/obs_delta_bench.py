"""Tracked against untracked observation stores on BASELINE config 3 (Knuffingen, 16384 envs, 480x640 classes, Stanley actions,
next-step autoreset): the same env alternates between the two every round (tc_track_obs on / off), so both legs run the same
build, the same envs and the same rollout. Per leg: env-steps/s from CUDA events around the timed steps, and the render kernel's
milliseconds per step from the library's own event timing (profile_begin / profile_end), the median SM clock and the peak
power nvidia-smi sampled during the leg, and the segments the leg's frames held (from the per-class segment export of one
untimed render at the leg's end). Then the 32-byte sectors a tracked step stores: the popcount of (old | new) mask words,
read from the library before and after a step, checked against the same count from the frames. Prints one JSON line.

    python tools/obs_delta_bench.py [--envs 16384] [--rounds 5] [--steps 100]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tinycarlo_b200 import TinyCarloVecEnv, _lib  # noqa: E402
from tinycarlo_b200.config import make_config  # noqa: E402
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "baseline"))
import workloads as WL  # noqa: E402
from bench import ClockSampler  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, sm = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:   # the device name alone still comes from torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("obs_delta_bench needs a CUDA device")
    info = {"card": card(), "library": _lib.build_info(), "envs": args.envs}
    print(json.dumps(info), flush=True)
    w = WL.WORKLOADS[3]
    cfg = make_config(w["map"], w["fmt"], car=w["car"], cam={"resolution": w["res"]})
    N = args.envs
    env = TinyCarloVecEnv(cfg, N, device="cuda:0", autoreset="next_step")
    speed = torch.full((N,), WL.STANLEY_SPEED, device="cuda:0")
    cc = torch.zeros((N, 2), device="cuda:0")
    man = torch.zeros(N, dtype=torch.int32, device="cuda:0")
    scale = 180.0 / np.pi / float(w["car"]["max_steering_angle"])

    def step():
        o = env.out
        cc[:, 0] = WL.STANLEY_SPEED
        cc[:, 1] = (o["heading_error"] + torch.atan2(WL.STANLEY_K * o["cte"], speed)) * scale
        env.step({"car_control": cc, "maneuver": man})

    def set_tracking(on):
        if on:
            env._track_obs, env._obs_seen = True, (None, None)   # the next step tracks self.obs again, all sectors dirty
        else:
            env._untrack_obs()

    seg_cnt = torch.zeros((N, env.n_classes), dtype=torch.int32, device="cuda:0")
    seg_i32 = torch.zeros((N, int(env.map.ll_edge_off[-1]), 4), dtype=torch.int32, device="cuda:0")

    def segments_per_frame():
        """segments drawn per frame at the current state: the unfused path's segment export, into a scratch frame buffer"""
        scratch = torch.empty_like(env.obs)
        _lib.check(env._L.tc_render(env._h, None, C.c_void_p(scratch.data_ptr()), _lib.TC_OBS_CLASSES, C.c_void_p(seg_cnt.data_ptr()),
                                    C.c_void_p(seg_i32.data_ptr()), env._stream()), "tc_render")
        torch.cuda.synchronize()
        del scratch
        return float(seg_cnt.sum()) / N

    env.reset(seed=0)
    for _ in range(10):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    legs = {"tracked": [], "untracked": []}
    for r in range(args.rounds):
        for name in ("tracked", "untracked"):
            set_tracking(name == "tracked")
            for _ in range(3):   # the first tracked step stores whole frames; leave it out of the window
                step()
            torch.cuda.synchronize()
            clocks = ClockSampler(0)
            clocks.start()
            env.profile_begin(args.steps)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            clk = clocks.stop()
            ms, k = env.profile_end()
            dt = e0.elapsed_time(e1)
            legs[name].append({"round": r, "env_steps_per_s": N * args.steps / (dt * 1e-3), "ms_per_step": dt / args.steps,
                               "render_ms": (ms["project"] + ms["raster"]) / max(k, 1), "track_ms": ms["track"] / max(k, 1),
                               "sm_mhz": clk.get("sm_mhz"), "power_w_max": clk.get("power_w_max"), "throttle": clk.get("reasons"),
                               "segments_per_env": segments_per_frame()})
            print(json.dumps({"leg": name, **legs[name][-1]}), flush=True)
    # sectors a tracked step stores: non-zero before or after the step
    set_tracking(True)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    words = env.obs_mask_words()
    m0 = torch.zeros(words, dtype=torch.int32, device="cuda:0")
    m1 = torch.zeros_like(m0)
    popcount8 = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.int64, device="cuda:0")
    popcount = lambda m: int(popcount8[m.view(torch.uint8).long()].sum())   # noqa: E731
    sec = lambda: env.obs.view(-1, 32).any(dim=1)   # noqa: E731
    counts, frame_counts = [], []
    for _ in range(10):
        env.obs_mask_words(m0)
        before = sec()
        step()
        env.obs_mask_words(m1)
        counts.append(popcount(m0 | m1))
        frame_counts.append(int((before | sec()).sum()))
        del before
    n_sec = env.obs.numel() // 32
    mask_bytes = n_sec // 8
    ratio = [t["env_steps_per_s"] / u["env_steps_per_s"] for t, u in zip(legs["tracked"], legs["untracked"])]
    out = dict(info)
    out.update({
        "tracked_env_steps_per_s": [x["env_steps_per_s"] for x in legs["tracked"]],
        "untracked_env_steps_per_s": [x["env_steps_per_s"] for x in legs["untracked"]],
        "speedup_per_round": ratio, "min_speedup": min(ratio),
        "render_ms_tracked": float(np.median([x["render_ms"] for x in legs["tracked"]])),
        "render_ms_untracked": float(np.median([x["render_ms"] for x in legs["untracked"]])),
        "sm_mhz_tracked": [x["sm_mhz"] for x in legs["tracked"]], "sm_mhz_untracked": [x["sm_mhz"] for x in legs["untracked"]],
        "segments_per_env_tracked": [x["segments_per_env"] for x in legs["tracked"]],
        "sectors_per_step": n_sec, "sectors_stored_per_step": counts, "mask_matches_frames": counts == frame_counts,
        "stored_fraction": float(np.mean(counts)) / n_sec,
        "stored_bytes_per_step": float(np.mean(counts)) * 32, "mask_bytes_read_per_step": mask_bytes,
        "cpu_oracle_fraction": "0.98-1.01 % (64 envs x 110 steps and 128 x 40 of the same workload)",
    })
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
