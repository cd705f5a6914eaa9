import os, sys, os.path as osp
sys.path.insert(0, '.'); sys.path.insert(0, 'tests')
import numpy as np, torch
from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv
cfg = {"num_executors": 10, "job_arrival_cap": 50, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0, "warmup_delay": 1000.0}
B = int(os.environ.get("POLICY_B", "4096"))  # 4096: mode 0 by default; up to 2 x SMs envs: mode 1
env = BatchedSparkSchedSimEnv(cfg, num_envs=B, decima_policy=True)
z = np.load(osp.join('tests', 'golden', 'decima_model.npz'))
env.set_decima_weights({k: z[k] for k in z.files})
env.reset_host((np.arange(B) + 5).astype(np.uint64))
env.set_autoreset(True, B)
env.rollout_decima(150)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for rep in range(3):
    e0.record()
    for _ in range(50): env.decima_policy()
    e1.record(); torch.cuda.synchronize()
    print("policy call: %.1f us" % (e0.elapsed_time(e1) * 1000 / 50))
e0.record(); env.rollout_decima(100); e1.record(); torch.cuda.synchronize()
print("rollout decision: %.1f us" % (e0.elapsed_time(e1) * 1000 / 100))
