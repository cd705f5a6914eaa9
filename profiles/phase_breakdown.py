"""Per-phase wall-cycle breakdown of the fused rollout, measured inside the kernel with clock64().

Needs the -DSSB_PROFILE build (built here as _lib/libssb_prof.so; ncu is not involved).  Usage on
the GPU box:  python profiles/phase_breakdown.py  [> profiles/rNN_phase_breakdown.txt]
"""
import ctypes as C
import os
import os.path as osp
import sys

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

import spark_sched_sim_b200.build as build  # noqa: E402

lib = os.environ.get("SSB_PROF_LIB") or osp.join(REPO, "spark-sched-sim_b200", "_lib", "libssb_prof.so")
if not osp.exists(lib):
    build.build(force=True, variant="prof", extra=["-DSSB_PROFILE"])
os.environ["SSB_LIB"] = lib

import torch  # noqa: E402

from spark_sched_sim_b200 import _native as nat  # noqa: E402
from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

SLOTS = {0: "fast loop (hot_load + batches + flush)", 2: "general-path events (pop_min + handle_event)",
         4: "schedulability scan / idle moves", 5: "take_action + end of round", 6: "reward",
         7: "observation", 8: "fair policy", 9: "owed graph + reward at the end of the launch",
         11: "  of which hot_load"}

cfg = {"num_executors": 10, "job_arrival_cap": 50, "job_arrival_rate": 4.0e-5,
       "moving_delay": 2000.0, "warmup_delay": 1000.0}
B = int(os.environ.get("SSB_PROF_B", "4096"))
env = BatchedSparkSchedSimEnv(cfg, num_envs=B)
env.reset_host((1234 + np.arange(B)).astype(np.uint64))
for _ in range(3):
    env.rollout_fair(128, True, True, B)
ptr = C.c_void_p()
nat.check(env.L.ssb_get_debug_counters(env._h, C.byref(ptr)), "ssb_get_debug_counters")
prof = env._view(ptr.value, B * 16 * 8, torch.int64).view(B, 16)
prof.zero_()
env.reset_stats()
torch.cuda.synchronize()
env.rollout_fair(128, True, True, B)
torch.cuda.synchronize()
p = prof.cpu().numpy().astype(np.float64)
st = env.stats()
total = p[:, 10].sum()
dec = st["decisions"]
print(f"# k_rollout_fair, {B} envs x 128 decisions; wall cycles per warp summed over envs; "
      f"events/decision = {st['events'] / dec:.1f}")
print(f"total cycles per decision per warp: {total / dec:,.0f}")
acc = 0.0
for k, name in SLOTS.items():
    if k != 11:
        acc += p[:, k].sum()
    print(f"{name:48s} {100 * p[:, k].sum() / total:6.2f} %   {p[:, k].sum() / dec:10,.0f} cycles/decision")
print(f"{'unattributed (loop control, resets)':48s} {100 * (total - acc) / total:6.2f} %")
print(f"fast iterations per decision: {p[:, 1].sum() / dec:.2f}   cycles per fast iteration: "
      f"{p[:, 0].sum() / max(p[:, 1].sum(), 1):,.0f}")
print(f"general-path events per decision: {p[:, 3].sum() / dec:.2f}   cycles per general-path event: "
      f"{p[:, 2].sum() / max(p[:, 3].sum(), 1):,.0f}")
