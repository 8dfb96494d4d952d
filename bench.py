#!/usr/bin/env python
"""bench.py — env-steps/s of the tinycarlo hot path on B200 (BASELINE.json metric), one JSON line on rank 0.

  python bench.py --gpus 1 --steps 100 --warmup 5                      # this repo's CUDA path, BASELINE config 3 (the metric's)
  python bench.py --config 2                                           # any of BASELINE.json's five configs (baseline/workloads.py)
  python bench.py --impl reference --steps 100 --warmup 5              # the CPU arm: the UNMODIFIED reference (baseline/_ref),
                                                                       #   one process per host core; C port of it as a second figure
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --steps 100 --warmup 5 --dump-outputs bench_outputs   # also writes what the last timed step returned, as .npy

Default workload (config.workload): BASELINE.json configs[2] — Knuffingen map, 480x640 `classes` observations (5x480x640 u8 =
1 536 000 B per env-step), Stanley-controller actions with lanepath CTE / heading info consumed every step, auto-reset of
finished envs; 16384 envs per GPU (weak scaling: per-GPU work is fixed, envs shard by index, no per-step collective; NCCL only
all-gathers episode statistics).

A "step" is one lockstep pass of the hot path over all envs of the rank. `value` is measured with the action tensors already on
the device (CUDA events on the launching stream, max over ranks) over exactly --steps steps; `sustained` (only with --min-seconds)
repeats that for a clock-determined number of steps; `e2e` drives the
same step from pinned HOST buffers (actions in, reward / flags / CTE / heading out, stream synchronised every step; observations
stay device-resident as the vectorised API defines); `e2e_obs_to_host` additionally brings the observations to the host
(bit-packed); `roofline` is the render kernel's algorithmic bytes over its own event-timed duration.

--dump-outputs DIR writes what the headline's last timed step returned to its caller (observations, reward, terminated,
truncated, every info tensor; rank 0's envs) as DIR/<name>.npy in float32 / float64, at most 64 MB in all. Inputs depend only on
the arguments (seeded resets and policy), so two builds of the library can be compared output for output.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the tree may be read-only: bench.py writes nothing into it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "baseline"))

import numpy as np  # noqa: E402
import workloads as WL  # noqa: E402  (baseline/workloads.py: plain data, no product / oracle imports)

UNIT = "env-steps/s"
SETUP = {}   # one-time set-up costs worth reporting (config 5: per-env camera parameters and their visible-set tables)


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def envs_per_gpu(w, args, world):
    if args.envs_per_gpu:
        return args.envs_per_gpu
    if w["scaling"] == "strong":
        return w["envs_total"] // world
    return w["envs_per_gpu"]


def config_dict(w, args, world):
    """The `config` object of the JSON line: identical in both arms (the driver compares them)."""
    n = envs_per_gpu(w, args, world)
    c = {"workload": f"{w['workload']}, {n} envs/GPU", "baseline_config": args.config, "envs_per_gpu": n, "envs_total": n * world,
         "obs_bytes_per_env_step": (WL.obs_bytes(w) if w["res"] else round(sum(WL.obs_bytes(w, r) for r in w["groups"]) / len(w["groups"]))),
         "l2": "observation tensors are far larger than L2 and written once per step; nothing is re-read between steps"}
    if graph_stepped(w, n):
        c["stepping"] = "policy ops + step captured once with TinyCarloVecEnv.capture() and replayed as a CUDA graph (launch-bound config); eager stepping is reported next to it"
    return c


def graph_stepped(w, n):
    """launch-bound configurations (a few thousand small frames, device-side random policy, no wrappers) are quoted as CUDA-graph replays"""
    return w["policy"] == "random" and not w.get("groups") and not w["wrappers"] and n <= 8192 and w["fmt"] == "classes"


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                                          str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)   # no sampler outlives a run that fails before stop()
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
                pw.append(float(p[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------------ CPU arms
def port_arm(w, n_envs, steps, warmup, threads, min_seconds=0.0):
    """The reference's algorithm restated in C (oracle/tc_oracle.c: the pinned oracle), all host threads via OpenMP, on the same
    workload. Runs `steps` lockstep passes, and keeps going until min_seconds have passed. -> (env-steps/s, seconds, passes).
    This is the only place besides tests/ and smoke() that executes oracle/ - as a measured baseline, never as the product."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    from oracle import oracle as orc
    from tinycarlo_b200.config import make_config   # a plain dict builder: nothing of the CUDA path is touched in this arm

    def oracle_env(cfg, n, wrapped=False, cam_rows=None, car_rows=None):
        omap = orc.load_named_map(cfg["map"]["map_name"], cfg["map"]["pixel_per_meter"], cfg["map"].get("spawn_points"))
        cc = cfg["camera"]
        H, W = cc["resolution"]
        if cam_rows is None:
            cam_rows = orc.pack_cam(*orc.camera_matrices(cc["position"], cc["orientation"], cc["fov"], [H, W]), cc["max_range"])
        if car_rows is None:
            car_rows = orc.pack_car(cfg["car"], cfg["sim"].get("fps", 30))
        return orc.OracleVecEnv(omap, n, car_rows, cam_rows, cc["line_thickness"], H, W, cfg["sim"]["observation_space_format"], wrapped=wrapped)
    reses = [w["res"]] if w["res"] else w["groups"]
    n_each = max(n_envs // len(reses), 1)
    envs, rngs = [], []
    p5 = WL.config5_params(w["envs_total"]) if w.get("groups") else None
    for gi, res in enumerate(reses):
        cfg = make_config(w["map"], w["fmt"], car=w["car"], cam={"resolution": res})
        cam_rows = car_rows = None
        if p5 is not None:
            ids = np.arange(gi * n_each, (gi + 1) * n_each)
            cam_rows = np.stack([orc.pack_cam(*orc.camera_matrices(p5["position"][i], p5["orientation"][i], p5["fov"][i], res), WL.CAM["max_range"])
                                 for i in ids])
            car_rows = np.tile(orc.pack_car(cfg["car"], 30), (n_each, 1))
            car_rows[:, 0], car_rows[:, 2], car_rows[:, 3] = p5["car"]["wheelbase"][ids], p5["car"]["max_velocity"][ids], p5["car"]["max_steering_angle"][ids]
        o = oracle_env(cfg, n_each, wrapped=bool(w["wrappers"]), cam_rows=cam_rows, car_rows=car_rows)
        r = [orc.make_rng(gi * n_each + i) for i in range(n_each)]
        o.reset([o.map.sample_spawn_node(x) for x in r])
        envs.append((o, cfg, car_rows))
        rngs.append(r)
    arng = np.random.default_rng(0)
    man = [np.zeros(n_each, np.int32) for _ in envs]
    ou = [np.zeros(n_each) for _ in envs]
    cnt = [np.zeros(n_each, np.int64) for _ in envs]
    state = {"t": 0}

    def one():
        for k, (o, cfg, car_rows) in enumerate(envs):
            max_steer = cfg["car"]["max_steering_angle"] if car_rows is None else car_rows[:, 3]
            if w["policy"] == "random":
                cc = arng.uniform(-1, 1, (n_each, 2)).astype(np.float32)
                man[k] = arng.integers(0, 4, n_each).astype(np.int32)
            else:
                steer = (o.heading_error + np.arctan2(WL.STANLEY_K * o.cte, WL.STANLEY_SPEED)) * 180 / np.pi / max_steer
                if w["policy"] == "stanley_ou_mixed":
                    if state["t"] % WL.MANEUVER_PERIOD == 0:
                        man[k] = arng.integers(0, 4, n_each).astype(np.int32)
                    ou[k] += WL.OU_THETA * (0.0 - ou[k]) + WL.OU_SIGMA * arng.standard_normal(n_each)
                    steer = np.clip(steer + ou[k], -1, 1)
                cc = np.stack([np.full(n_each, WL.STANLEY_SPEED), steer], 1).astype(np.float32)
            o.step(cc.astype(np.float64), man[k])
            done = (o.terminated | o.truncated).astype(bool)
            for name, kw in w["wrappers"]:   # the wrappers' arithmetic on the info arrays (reward.py:44-62, termination.py:24-48)
                if name == "CTETerminationWrapper":
                    over = np.abs(o.cte) > kw["max_cte"]
                    cnt[k] = np.where(over, cnt[k] + 1, 0)
                    fire = cnt[k] >= kw["number_of_steps"]
                    cnt[k][fire] = 0
                    done |= fire
            if done.any():
                o.reset([o.map.sample_spawn_node(r) if d else 0 for r, d in zip(rngs[k], done)], mask=done)
        state["t"] += 1
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    done_steps = 0
    while done_steps < steps or time.perf_counter() - t0 < min_seconds:
        one()
        done_steps += 1
    dt = time.perf_counter() - t0
    return n_each * len(envs) * done_steps / dt, dt, done_steps


def reference_sample(w, procs, seconds):
    """A bounded sample of the unmodified reference: calibrates one process first (that is also the single-process figure),
    then runs `procs` processes for about `seconds`. -> dict for cpu_baseline, or None when baseline/_ref is absent."""
    import ref_arm
    if not ref_arm.available():
        return None
    single, s_dt, _ = ref_arm.run(w, 1, 3, 40)
    n = max(int(single * seconds * 0.8), 20)   # co-running processes are somewhat slower than one alone
    agg, dt, per = ref_arm.run(w, procs, 3, n)
    return {"value": agg, "unit": UNIT, "cores": procs, "kind": "reference",
            "sample": f"unmodified reference (baseline/_ref, gym.make('tinycarlo-v2') loop), {procs} processes x {n} env-steps of the same workload ({dt:.1f} s)",
            "single_process": {"value": single, "sample": f"1 process x 40 env-steps ({s_dt:.1f} s)"},
            "cpu_model": ref_arm.cpu_model(), "versions": ref_arm.versions()}


def reference_main(args, w, rank, world):
    """--impl reference: rank 0 only. One "step" = every host core advancing its own reference env by S env-steps."""
    if rank != 0:
        return
    import ref_arm
    threads = host_threads()
    W = max(args.warmup, 1)
    line = {"impl": "reference", "metric": w["metric"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": W,
            "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(w, args, world), "gpu_launches": 0}
    port_n = args.cpu_envs or min(128 * threads, 2048)
    if w.get("groups"):
        port_n = min(port_n, 96 * threads)
    if ref_arm.available():
        S = max(1, min(8, 1200 // max(args.steps, 1)))           # env-steps per process per bench "step": the run stays within minutes
        val, dt, per = ref_arm.run(w, threads, W * S, args.steps * S)
        single, s_dt, _ = ref_arm.run(w, 1, 3, 60)
        pval, pdt, ppass = port_arm(w, port_n, 4, 1, threads, min_seconds=min(args.cpu_seconds, 8.0))
        line.update({"value": val, "ms_per_step": dt / args.steps * 1e3,
                     "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "reference",
                                      "sample": f"unmodified reference from baseline/_ref through gym.make('tinycarlo-v2') + env.step, {threads} processes x "
                                                f"{args.steps} steps x {S} env-steps ({dt:.1f} s)",
                                      "single_process": {"value": single, "sample": f"1 process x 60 env-steps ({s_dt:.1f} s)"},
                                      "cpu_model": ref_arm.cpu_model(), "versions": ref_arm.versions()},
                     "cpu_baseline_port": {"value": pval, "unit": UNIT, "cores": threads, "kind": "port",
                                           "sample": f"{port_n} envs x {ppass} lockstep steps, oracle/tc_oracle.c with OpenMP ({pdt:.1f} s)"}})
    else:
        # baseline/_ref did not travel (it is built by __graft_entry__.build() where /root/reference exists): the C port stands in
        val, dt, _ = port_arm(w, port_n, args.steps, W, threads)
        line.update({"value": val, "ms_per_step": dt / args.steps * 1e3,
                     "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                                      "sample": f"baseline/_ref absent; {port_n} envs x {args.steps} lockstep steps ({dt:.1f} s), oracle/tc_oracle.c with OpenMP"}})
    line["e2e"] = {"value": line["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ this repo's arm
def build_env(w, N, dev, rank, world):
    """-> (env to step, list of base TinyCarloVecEnv handles, per-env max steering angle or float)"""
    import torch
    from tinycarlo_b200 import TinyCarloGroupedVecEnv, TinyCarloVecEnv
    from tinycarlo_b200.config import make_config
    from tinycarlo_b200.distributed import shard_groups
    from tinycarlo_b200 import wrapper as wrappers
    max_steer = float(w["car"]["max_steering_angle"])
    if w.get("groups"):
        total = N * world
        sizes, offs = shard_groups(WL.group_sizes(total), rank, world)
        cfg = make_config(w["map"], w["fmt"], car=w["car"])
        env = TinyCarloGroupedVecEnv(cfg, list(zip(sizes, w["groups"])), device=dev, group_index_offsets=offs, autoreset="next_step")
        p = WL.config5_params(total)
        ms = []
        t0 = time.perf_counter()
        for e, n, o in zip(env.envs, sizes, offs):
            sl = slice(o, o + n)
            e.set_camera_params(position=p["position"][sl], orientation=p["orientation"][sl], fov=p["fov"][sl])
            e.set_car_params(**{k: v[sl] for k, v in p["car"].items()})
            ms.append(torch.from_numpy(p["car"]["max_steering_angle"][sl]).to(dev, torch.float32))
        # one-time cost of per-env camera parameters: E / K of every env on the host (the reference's cv2.Rodrigues / numpy calls,
        # for bit parity) plus the visible-set tables of each group, built once per camera reach and cached by the library
        SETUP["set_params_s"] = time.perf_counter() - t0
        SETUP["visible_set_tables"] = [e.cull_stats() for e in env.envs]
        return env, env.envs, torch.cat(ms)
    cfg = make_config(w["map"], w["fmt"], car=w["car"], cam={"resolution": w["res"]})
    base = TinyCarloVecEnv(cfg, N, device=dev, env_index_offset=rank * N, autoreset="next_step")
    env = base
    for name, kw in w["wrappers"]:
        env = getattr(wrappers, name)(env, **kw)
    return env, [base], max_steer


DUMP_BUDGET = {"obs": 47_000_000, "rest": 16_000_000}   # bytes; with the .npy headers the whole dump stays under 64 MB


def sample_outputs(ret):
    """Host copies of what env.step() returned -> {name: ndarray}: obs (obs_g<i> per resolution group), reward, terminated,
    truncated, info_<key>. float64 data and 32/64-bit integers become float64, everything else float32 (both exact). An array
    over its share of the budget keeps a fixed, seeded sample of its envs (dim 0), whose indices are stored as <name>_rows."""
    import torch
    obs, reward, term, trunc, info = ret
    groups = {"obs": obs} if torch.is_tensor(obs) else {f"obs_g{i}": o for i, o in enumerate(obs)}
    rest = {"reward": reward, "terminated": term, "truncated": trunc, **{f"info_{k}": v for k, v in info.items()}}
    out = {}
    for part, arrays in (("obs", groups), ("rest", rest)):
        share = DUMP_BUDGET[part] // len(arrays)
        for name, t in arrays.items():
            dt = torch.float64 if t.dtype in (torch.float64, torch.int32, torch.int64) else torch.float32
            n = t.shape[0]
            row_bytes = (t.numel() // max(n, 1)) * dt.itemsize
            k = min(n, max(share // (row_bytes + 8), 1))
            if k < n:
                rows = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
                t = t[torch.from_numpy(rows).to(t.device)]
                out[name + "_rows"] = rows.astype(np.float64)
            out[name] = t.to(dt).cpu().numpy()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[1, 2, 3, 4, 5], help="BASELINE.json config (1-based); 3 is the one the metric is quoted on")
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="override the config's env count per GPU")
    ap.add_argument("--graph-steps", type=int, default=5, help="env steps captured per CUDA-graph replay (launch-bound configs)")
    ap.add_argument("--min-seconds", type=float, default=0.0, help="length of a sustained device-timed run reported next to the K-step one "
                    "(0: none, so that --steps alone sets how many steps are timed)")
    ap.add_argument("--cpu-envs", type=int, default=0, help="envs of the C-port sample (default: 128 x host threads, at most 2048: 3 GB of frames)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="length of the cpu_baseline samples")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-fill-context", action="store_true", help="skip the memset / zero-fill context numbers (keeps ncu launch lists clean)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the CUDA arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = WL.WORKLOADS[args.config]
    if args.impl == "reference":
        return reference_main(args, w, rank, world)

    import torch
    import torch.distributed as dist
    from tinycarlo_b200 import _lib
    from tinycarlo_b200.distributed import EpisodeStats
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N = envs_per_gpu(w, args, world)
    env, bases, max_steer = build_env(w, N, dev, rank, world)
    grouped = len(bases) > 1
    torch.manual_seed(1000 + rank)
    cc = torch.zeros((N, 2), dtype=torch.float32, device=dev)
    maneuver = torch.zeros(N, dtype=torch.int32, device=dev)
    ou = torch.zeros(N, device=dev)
    speed_t = torch.full((N,), WL.STANLEY_SPEED, device=dev)
    stats = EpisodeStats(dev)
    state = {"t": 0, "info": None, "gathered": None}
    steer_scale = 180.0 / np.pi / max_steer
    policy = w["policy"]

    _, info0 = env.reset(seed=0)
    state["info"] = info0

    def act():
        if policy == "random":      # examples/random_control.py:11 on the device
            cc.uniform_(-1.0, 1.0)
            maneuver.random_(0, 4)
        else:                       # examples/stanley_control.py:56-58 as tensor ops on the info of the previous step
            i = state["info"]
            cc[:, 0] = WL.STANLEY_SPEED
            steer = (i["heading_error"] + torch.atan2(WL.STANLEY_K * i["cte"], speed_t)) * steer_scale
            if policy == "stanley_ou_mixed":
                if state["t"] % WL.MANEUVER_PERIOD == 0:
                    maneuver.random_(0, 4)
                ou.add_(-WL.OU_THETA * ou + WL.OU_SIGMA * torch.randn_like(ou))
                steer = (steer + ou).clamp_(-1.0, 1.0)
            cc[:, 1] = steer
        return {"car_control": cc, "maneuver": maneuver}

    def step_device():
        state["ret"] = env.step(act())
        _, reward, term, trunc, info = state["ret"]
        state["info"] = info
        stats.update(reward, term, trunc)
        state["t"] += 1
        if w["wrappers"] and state["t"] % 100 == 0:
            state["gathered"] = stats.gather()      # config 4: per-rank episode statistics over NCCL every 100 steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def launches():
        return sum(b.launch_count for b in bases)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()   # sampled from the warm-up to the end of the device-timed regions (all under load)
    W = max(args.warmup, 3)
    for _ in range(W):
        step_device()
    barrier()
    l0 = launches()
    if not grouped:
        bases[0].profile_begin(args.steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_device()
    if world > 1:
        state["gathered"] = stats.gather()     # episode statistics over NVLink: the only collective
    e1.record()
    barrier()
    elapsed_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    n_launch = launches() - l0
    kern = {}
    if not grouped:
        kern_ms, kern_steps = bases[0].profile_end()
        kern = {k: v / max(kern_steps, 1) for k, v in kern_ms.items()}
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(elapsed_ms.item()) / args.steps
    value = N * world / (ms_per_step * 1e-3)
    dump = None
    if args.dump_outputs and rank == 0 and not graph_stepped(w, N):
        dump = sample_outputs(state["ret"])

    # ---- launch-bound configs: the policy + step captured in a CUDA graph (TinyCarloVecEnv.capture), replayed. It runs before
    # the clock-determined sustained loop, so that its last step, the headline's, depends on the arguments only.
    graph = None
    if graph_stepped(w, N):
        per = args.graph_steps if args.graph_steps > 0 and args.steps % args.graph_steps == 0 else 1   # env steps per replay; K stays exact
        g = bases[0].capture(lambda e: act(), steps=per)
        for _ in range(3):
            g.replay()
        barrier()
        e0.record()
        for _ in range(args.steps // per):
            g.replay()
        e1.record()
        barrier()
        g_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(g_ms, op=dist.ReduceOp.MAX)
        graph = {"value": N * world * args.steps / (float(g_ms.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(g_ms.item()) / args.steps,
                 "note": f"policy ops + step captured once with TinyCarloVecEnv.capture(steps={per}) and replayed: one graph launch per {per} step(s)"}
        if args.dump_outputs and rank == 0:   # the replays wrote into the buffers the eager step returned views of
            dump = sample_outputs(state["ret"])

    # ---- the same loop for at least --min-seconds (clocks and power settle): the sustained figure
    sustained = None
    if args.min_seconds > 0:
        chunk = max(args.steps, 10)
        n_chunks = max(int(np.ceil(args.min_seconds * 1e3 / (ms_per_step * chunk))), 1)
        barrier()
        e0.record()
        for _ in range(n_chunks * chunk):
            step_device()
        e1.record()
        barrier()
        s_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(s_ms, op=dist.ReduceOp.MAX)
        sustained = {"value": N * world * n_chunks * chunk / (float(s_ms.item()) * 1e-3), "unit": UNIT, "seconds": float(s_ms.item()) * 1e-3,
                     "steps": n_chunks * chunk}
    clocks = sampler.stop() if rank == 0 else None

    # ---- config 5: per-group kernel times from a serial pass (the groups normally overlap on separate streams)
    group_rows = None
    if grouped:
        env.overlap = False
        for b in bases:
            b.profile_begin(20)
        for _ in range(20):
            step_device()
        torch.cuda.synchronize(dev)
        group_rows = []
        for b, res in zip(bases, w["groups"]):
            km, ks = b.profile_end()
            group_rows.append({"res": res, "envs": b.num_envs, "obs_bytes": b.obs.numel(), "track_ms": km["track"] / max(ks, 1),
                               "render_ms": (km["project"] + km["raster"]) / max(ks, 1)})
        env.overlap = True

    # ---- end to end from pinned host buffers: actions in, reward / flags / cte / heading out, synchronised every step
    e2e = None
    if not args.no_e2e:
        pin = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt).pin_memory()   # noqa: E731
        h_cc, h_man = pin(N, 2), pin(N, dt=torch.int32)
        h_rew, h_cte, h_head = pin(N), pin(N), pin(N)
        h_term, h_trunc = pin(N, dt=torch.uint8), pin(N, dt=torch.uint8)
        h_cc[:, 0] = WL.STANLEY_SPEED
        cc_np, man_np, cte_np, head_np = h_cc.numpy(), h_man.numpy(), h_cte.numpy(), h_head.numpy()
        hrng = np.random.default_rng(rank)
        ms_np = max_steer.cpu().numpy() if torch.is_tensor(max_steer) else max_steer
        ou_np = np.zeros(N, np.float32)
        plain = not grouped and not w["wrappers"]
        hstate = {"t": 0}

        def step_host():
            if policy == "random":
                cc_np[:] = hrng.uniform(-1, 1, (N, 2))
                man_np[:] = hrng.integers(0, 4, N)
            else:
                steer = (head_np + np.arctan2(WL.STANLEY_K * cte_np, WL.STANLEY_SPEED)) * (180.0 / np.pi / ms_np)
                if policy == "stanley_ou_mixed":
                    if hstate["t"] % WL.MANEUVER_PERIOD == 0:
                        man_np[:] = hrng.integers(0, 4, N)
                    ou_np[:] += -WL.OU_THETA * ou_np + WL.OU_SIGMA * hrng.standard_normal(N).astype(np.float32)
                    steer = np.clip(steer + ou_np, -1, 1)
                cc_np[:, 1] = steer
            hstate["t"] += 1
            if plain:   # the C ABI's host-buffer entry point does the copies and the synchronisation itself
                bases[0].step_host(h_cc, h_man, h_rew, h_term, h_trunc, h_cte, h_head)
            else:       # wrappers / groups sit above the ABI: the same copies through torch
                cc.copy_(h_cc, non_blocking=True)
                maneuver.copy_(h_man, non_blocking=True)
                _, reward, term, trunc, info = env.step({"car_control": cc, "maneuver": maneuver})
                h_rew.copy_(reward, non_blocking=True)
                h_term.copy_(term.view(torch.uint8), non_blocking=True)
                h_trunc.copy_(trunc.view(torch.uint8), non_blocking=True)
                h_cte.copy_(info["cte"], non_blocking=True)
                h_head.copy_(info["heading_error"], non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
        for _ in range(2):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host()
        torch.cuda.synchronize(dev)
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": N * world * args.steps / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": N * 12,
               "d2h_bytes_per_step": N * 14, "note": ("tc_step_host" if plain else "torch copies around env.step") + ": pinned host actions in, "
               "reward/terminated/truncated/cte/heading out, stream synchronised every step; observations stay in HBM (the vectorised entry point returns CUDA tensors)"}

    # ---- context next to the copy peak: the driver's memset and torch's fill of the same observation tensor (pure-write ceilings)
    fill = {}
    if not args.no_fill_context and not grouped:
        obs = bases[0].obs
        nbytes = obs.numel() * obs.element_size()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = 0.0
        for _ in range(3):
            w0.record()
            obs.zero_()
            w1.record()
            torch.cuda.synchronize(dev)
            best = max(best, nbytes / (w0.elapsed_time(w1) * 1e-3) / 1e9)
        fill["torch_zero_fill_gbs"] = best
        try:
            import ctypes
            rt = None
            for name in ("libcudart.so", "libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
                try:
                    rt = ctypes.CDLL(name)
                    break
                except OSError:
                    continue
            if rt is not None:
                rt.cudaMemsetAsync.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p]
                stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                best = 0.0
                for _ in range(3):
                    w0.record()
                    rc = rt.cudaMemsetAsync(ctypes.c_void_p(obs.data_ptr()), 0, nbytes, stream)
                    w1.record()
                    torch.cuda.synchronize(dev)
                    if rc == 0:
                        best = max(best, nbytes / (w0.elapsed_time(w1) * 1e-3) / 1e9)
                fill["cuda_memset_gbs"] = best or None
        except Exception:
            pass

    # ---- observations to the HOST every step (what a CPU-side consumer pays): bit-packed frames, one D2H copy per step
    e2e_obs = None
    if not args.no_e2e and rank == 0 and not grouped and w["fmt"] == "classes":
        e2e_obs = obs_to_host_leg(w, dev, args, max_steer)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (rasterise + store): algorithmic bytes = the observation, written once
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    so_hash = _lib.build_info()
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        ent = tj["configs"].get(str(args.config))
        if ent:
            match = ent.get("so_hash") == so_hash
            traffic_src = {"file": "profiles/traffic.json", "so_hash": ent.get("so_hash"), "matches_loaded_library": match,
                           "dram_bytes_per_env": ent["dram_bytes_per_env"], "capture": ent.get("capture")}
            if match:
                traffic = ent["dram_bytes_per_env"] * N
    except Exception:
        pass
    def kernel_name(b):
        """the render kernel a handle launches (tc_debug_render_info)"""
        ri = b.render_info()
        fmt = {"rgb": "RGB", "classes_bits": "BITS", "classes_bf16": "BF16"}.get(b.observation_space_format, "U8")
        if ri["block_per_env"]:
            return f"tc_render_envs_kernel<256,{fmt},{ri['envs_per_block']}>" if ri["envs_per_block"] else f"tc_render_env_kernel<256,{fmt}>"
        if fmt in ("RGB", "BITS") and ri["banded_smem"]:
            return "tc_prims_kernel + tc_draw_class_kernel<BITS>" if fmt == "BITS" else "tc_render_env_banded_kernel<RGB>"
        return f"tc_render_classes_kernel<256,{fmt}>"
    if grouped:
        for r, b in zip(group_rows, bases):
            r["achieved_gbs"] = r["obs_bytes"] / (r["render_ms"] * 1e-3) / 1e9 if r["render_ms"] > 0 else 0.0
            r["kernel"] = kernel_name(b)
        top = max(group_rows, key=lambda r: r["render_ms"])
        raster_ms, alg_bytes = top["render_ms"], top["obs_bytes"]
        kname = top["kernel"] + f" ({top['res'][0]}x{top['res'][1]} group)"
    else:
        raster_ms = kern["project"] + kern["raster"] if kern.get("project", 0) > 0.01 * max(kern["raster"], 1e-9) else kern["raster"]
        alg_bytes = bases[0].obs.numel() * bases[0].obs.element_size()
        kname = kernel_name(bases[0])
    achieved = alg_bytes / (raster_ms * 1e-3) / 1e9 if raster_ms > 0 else 0.0
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "algorithmic_bytes": alg_bytes, "kernel": kname, "kernel_ms_per_launch": raster_ms,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "step_share_ms": kern or None, "groups": group_rows, "frac_of_nominal_8tbs": achieved / 8000.0, **fill}

    cpu_baseline = cpu_port = None
    if not args.no_cpu_baseline and world == 1:
        threads = host_threads()
        cpu_baseline = reference_sample(w, threads, args.cpu_seconds)
        n_cpu = args.cpu_envs or min(128 * threads, 2048)
        if grouped:
            n_cpu = min(n_cpu, 96 * threads)
        val, dt, passes = port_arm(w, n_cpu, 4, 1, threads, min_seconds=min(args.cpu_seconds, 8.0))
        cpu_port = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": f"{n_cpu} envs x {passes} lockstep steps of the same workload, oracle/tc_oracle.c with OpenMP ({dt:.1f} s)"}
        if cpu_baseline is None:
            cpu_baseline, cpu_port = cpu_port, None

    obs_b = sum(b.obs.numel() * b.obs.element_size() for b in bases)
    gathered = state["gathered"]
    st = (gathered.sum(0) if gathered is not None else stats.local).tolist()
    eager = None
    if graph is not None:   # the headline of a launch-bound config is the graph replay; the eager loop stays in the line
        eager = {"value": value, "unit": UNIT, "ms_per_step": ms_per_step}
        value, ms_per_step = graph["value"], graph["ms_per_step"]
    line = {"metric": w["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms_per_step, "eager": eager, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_dict(w, args, world), "obs_gbs": value / (N * world) * obs_b * world / 1e9,
            "sustained": sustained, "cuda_graph": graph, "clocks": clocks, "e2e": e2e, "e2e_obs_to_host": e2e_obs, "gpu_launches": n_launch,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "cpu_baseline_port": cpu_port, "library": {"so_hash": so_hash}, "setup": SETUP or None,
            "episode_stats": {"finished": st[0], "truncated": st[1], "reward_sum": st[2], "env_steps": st[3]}}
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def obs_to_host_leg(w, dev, args, max_steer):
    """Host loop WITH the observations brought to pinned host memory every step: 1 bit per pixel frames (classes_bits: 8x fewer
    bytes than u8, nothing lost) through TinyCarloVecEnv.step_host(obs_host=...), one D2H copy per step."""
    import torch
    from tinycarlo_b200 import TinyCarloVecEnv
    from tinycarlo_b200.config import make_config
    n = min(w["envs_per_gpu"], 4096)
    cfg = make_config(w["map"], w["fmt"], car=w["car"], cam={"resolution": w["res"]})
    try:
        env = TinyCarloVecEnv(cfg, n, device=dev, autoreset="next_step", obs_format="classes_bits")
        env.reset(seed=0)
    except Exception as e:   # e.g. H*W not a multiple of 32 (84x84)
        return {"unavailable": str(e)}
    pin = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt).pin_memory()   # noqa: E731
    h_obs = torch.zeros(env.obs.shape, dtype=env.obs.dtype).pin_memory()
    hs = [pin(n, 2), pin(n, dt=torch.int32), pin(n), pin(n, dt=torch.uint8), pin(n, dt=torch.uint8), pin(n), pin(n)]
    hs[0][:, 0] = WL.STANLEY_SPEED
    rng = np.random.default_rng(0)
    ms = float(max_steer) if not torch.is_tensor(max_steer) else 30.0

    def one():
        if w["policy"] == "random":
            hs[0].numpy()[:] = rng.uniform(-1, 1, (n, 2))
            hs[1].numpy()[:] = rng.integers(0, 4, n)
        else:
            hs[0].numpy()[:, 1] = (hs[6].numpy() + np.arctan2(WL.STANLEY_K * hs[5].numpy(), WL.STANLEY_SPEED)) * (180.0 / np.pi / ms)
        env.step_host(*hs, obs_host=h_obs)
    for _ in range(3):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    dt = time.perf_counter() - t0
    nb = int(h_obs.numel() * h_obs.element_size())
    out = {"value": n * args.steps / dt, "unit": UNIT, "envs": n, "h2d_bytes_per_step": n * 12, "d2h_bytes_per_step": n * 14 + nb,
           "pcie_gbs": nb * args.steps / dt / 1e9, "nonzero_pixels": int((h_obs != 0).sum().item() > 0),
           "note": "as e2e, plus the observations copied to pinned host memory every step as 1 bit per pixel (classes_bits)"}
    env.close()
    return out


if __name__ == "__main__":
    main()
