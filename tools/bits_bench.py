"""Knuffingen 480x640 as 1 bit per pixel (obs_format="classes_bits"), 16384 envs: step and per-kernel times."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from tinycarlo_b200 import TinyCarloVecEnv
from tinycarlo_b200.config import make_config

n = int(os.environ.get("TC_ENVS", 16384))
cfg = make_config("knuffingen", "classes", cam={"resolution": [480, 640]})
env = TinyCarloVecEnv(cfg, n, device="cuda:0", autoreset="next_step", obs_format=os.environ.get("TC_FMT", "classes_bits"))
env.reset(seed=0)
cc = torch.zeros((n, 2), device="cuda"); man = torch.zeros(n, dtype=torch.int32, device="cuda")


def one():
    o = env.out
    cc[:, 0] = 0.8
    cc[:, 1] = (o["heading_error"] + torch.atan2(4 * o["cte"], torch.full_like(o["cte"], 0.8))) * (180 / np.pi / 30)
    env.step({"car_control": cc, "maneuver": man})


for _ in range(10):
    one()
torch.cuda.synchronize()
steps = 40
env.profile_begin(steps)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(steps):
    one()
e1.record(); torch.cuda.synchronize()
k, ks = env.profile_end()
ms = e0.elapsed_time(e1) / steps
nb = env.obs[0].numel() * env.obs.element_size()
print(f"N={n} step {ms:.3f} ms track {k['track'] / ks:.3f} render {(k['project'] + k['raster']) / ks:.3f}  -> {n / ms / 1e3:.2f} M env-steps/s  "
      f"{n * nb / ms / 1e6:.0f} GB/s  set pixels per env {int((env.obs != 0).sum().item()) / n:.0f} words")
